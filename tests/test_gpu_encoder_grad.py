"""GPU (B200): fine-tuning the encoder -- autograd through VisionTransformer.forward_feats / forward / get_intermediate_layers
(vitocm_encoder_train_forward / vitocm_encoder_backward) against torch.autograd over the float64 functional forward of
oracle/vit_oracle.py, for every parameter and the input."""
from functools import partial

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import vitocm_b200 as vob
from conftest import load_golden
from encoder_grad_cases import CASES, N_CLASSES, inputs as _inputs, loss as _loss, oracle_feats as _oracle_feats
from oracle import vit_oracle as VO

pytestmark = pytest.mark.gpu

# the bars tests/test_gpu_train.py holds the MIM step to: global relative L2 error over all gradients, and per tensor the largest
# error relative to the tensor's largest entry
GRAD_TOL_GLOBAL = 3e-2
GRAD_TOL_TENSOR = 2e-1

def _model(cfg, sd, precision):
    m = vob.VisionTransformer(img_size=[cfg.img_size], patch_size=cfg.patch_size, embed_dim=cfg.embed_dim, depth=cfg.depth,
                              num_heads=cfg.num_heads, mlp_ratio=cfg.mlp_ratio, qkv_bias=True,
                              norm_layer=partial(torch.nn.LayerNorm, eps=cfg.eps), precision=precision)
    m.load_state_dict(sd, strict=True)
    return m.cuda().train()


def _oracle_grads(sd, cfg, x, upstream, u):
    leaves = {k: v.detach().double().cuda().requires_grad_(True) for k, v in sd.items()}
    xd = x.double().cuda().requires_grad_(True)
    loss = _loss(upstream, lambda: _oracle_feats(leaves, cfg, xd, 1)[0], lambda: _oracle_feats(leaves, cfg, xd, 1)[0][:, 0],
                 lambda: _oracle_feats(leaves, cfg, xd, 4), u, torch.float64, "cuda")
    loss.backward()
    return {k: v.grad for k, v in leaves.items()}, xd.grad


def _errors(model, ref, x_grad, ref_dx):
    num = den = 0.0
    worst = (0.0, "")
    for n, p in model.named_parameters():
        r = ref[n]
        assert p.grad is not None, n
        d = (p.grad.double() - r).reshape(-1)
        num += float(d.pow(2).sum())
        den += float(r.pow(2).sum())
        worst = max(worst, (float(d.abs().max() / r.abs().max().clamp_min(1e-30)), n))
    dx_rel = float((x_grad.double() - ref_dx).norm() / ref_dx.norm())
    dx_max = float((x_grad.double() - ref_dx).abs().max() / ref_dx.abs().max())
    return (num / den) ** 0.5, worst, dx_rel, dx_max


@pytest.mark.parametrize("upstream", ["head", "feats", "intermediate"])
@pytest.mark.parametrize("case", list(CASES))
def test_gradients_match_float64_oracle(case, upstream):
    cfg, H, W, B = CASES[case]
    sd = VO.randomize_affine(VO.init_state_dict(cfg, seed=21), seed=22)
    x, u = _inputs(cfg, H, W, B, seed=23)
    ref, ref_dx = _oracle_grads(sd, cfg, x, upstream, u)
    for precision in ("bf16", "fp16"):
        m = _model(cfg, sd, precision)
        xc = x.cuda().requires_grad_(True)
        loss = _loss(upstream, lambda: m.forward_feats(xc), lambda: m(xc), lambda: m.get_intermediate_layers(xc, n=4), u,
                     torch.float32, "cuda")
        loss.backward()
        assert xc.grad is not None and xc.grad.shape == x.shape and xc.grad.dtype == torch.float32
        g, worst, dx_rel, dx_max = _errors(m, ref, xc.grad, ref_dx)
        print(f"{case} {upstream} {precision}: global relative L2 {g:.3e}, worst tensor {worst[0]:.3e} ({worst[1]}), "
              f"dx relative L2 {dx_rel:.3e}, dx max {dx_max:.3e}")
        assert g <= GRAD_TOL_GLOBAL, (precision, g)
        assert worst[0] <= GRAD_TOL_TENSOR, (precision, worst)
        assert dx_rel <= GRAD_TOL_GLOBAL and dx_max <= GRAD_TOL_TENSOR, (precision, dx_rel, dx_max)
        del m


def _tiny(precision, seed=31):
    cfg, H, W, B = CASES["tiny-48x64"]
    sd = VO.randomize_affine(VO.init_state_dict(cfg, seed=seed), seed=seed + 1)
    x, u = _inputs(cfg, H, W, B, seed=seed + 2)
    return _model(cfg, sd, precision), x.cuda(), u["r_feats"].cuda(), cfg, sd


def _grads(m, x, r, scale):
    m.zero_grad(set_to_none=True)
    xc = x.clone().requires_grad_(True)
    (m.forward_feats(xc) * (r * scale)).sum().backward()
    return torch.cat([p.grad.reshape(-1) for p in m.parameters()] + [xc.grad.reshape(-1)])


def test_fp16_power_of_two_upstream_scales_every_gradient_exactly():
    """fp16: S follows max |dfeats|'s exponent, so 2^k times the upstream gives 2^k times every gradient -- up to the run-to-run
    ordering of the fp32 atomic reductions, measured here by repeating the unscaled call.  A zero upstream gives exact zeros."""
    m, x, r, _, _ = _tiny("fp16")
    g0 = _grads(m, x, r, 1.0)
    spread = (_grads(m, x, r, 1.0) - g0).abs().max().item()
    for k in (-20, -6, 5, 12):
        gk = _grads(m, x, r, 2.0 ** k)
        diff = (gk / 2.0 ** k - g0).abs().max().item()
        assert diff <= 2 * spread + 1e-7 * g0.abs().max().item(), (k, diff, spread)
    for precision in ("fp16", "bf16"):
        mz, xz, rz, _, _ = _tiny(precision)
        gz = _grads(mz, xz, rz, 0.0)
        assert torch.equal(gz, torch.zeros_like(gz)), precision


def _grads_inter(m, x, rs, scale):
    m.zero_grad(set_to_none=True)
    xc = x.clone().requires_grad_(True)
    sum((f * (r * scale)).sum() for f, r in zip(m.get_intermediate_layers(xc, n=len(rs)), rs)).backward()
    return torch.cat([p.grad.reshape(-1) for p in m.parameters()] + [xc.grad.reshape(-1)])


def test_fp16_loss_scale_follows_the_largest_upstream_over_every_intermediate_layer():
    """get_intermediate_layers(n=3) with the largest |dfeats| in the FIRST slab: S must come from all slabs (a scale from the last
    slab alone would overflow fp16 there, or lose the power-of-two exactness).  Checked against the float64 oracle and for
    2^k exactness as above."""
    m, x, r, cfg, sd = _tiny("fp16")
    g = torch.Generator().manual_seed(5)
    rs = [torch.randn(r.shape, generator=g).cuda() * s for s in (2.0 ** 12, 1.0, 2.0 ** -3)]
    g0 = _grads_inter(m, x, rs, 1.0)
    assert torch.isfinite(g0).all()
    spread = (_grads_inter(m, x, rs, 1.0) - g0).abs().max().item()
    for k in (-8, 3):
        diff = (_grads_inter(m, x, rs, 2.0 ** k) / 2.0 ** k - g0).abs().max().item()
        assert diff <= 2 * spread + 1e-7 * g0.abs().max().item(), (k, diff, spread)
    leaves = {k: v.detach().double().cuda().requires_grad_(True) for k, v in sd.items()}
    xd = x.double().requires_grad_(True)
    sum((f * r.double()).sum() for f, r in zip(_oracle_feats(leaves, cfg, xd, 3), rs)).backward()
    ref = torch.cat([leaves[n].grad.reshape(-1) for n, _ in m.named_parameters()] + [xd.grad.reshape(-1)])
    assert float((g0.double() - ref).norm() / ref.norm()) <= GRAD_TOL_GLOBAL


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_gradient_accumulation_over_two_backwards(precision):
    m, x, r, _, _ = _tiny(precision)
    g1 = _grads(m, x, r, 1.0)
    g2 = _grads(m, x.flip(0), r, 1.0)
    m.zero_grad(set_to_none=True)
    for xb in (x, x.flip(0)):                      # forward -> backward per micro-batch
        (m.forward_feats(xb) * r).sum().backward()
    acc = torch.cat([p.grad.reshape(-1) for p in m.parameters()])
    want = (g1 + g2)[:acc.numel()]
    assert (acc - want).abs().max().item() <= 1e-5 * want.abs().max().item()


def test_overwritten_activations_raise():
    m, x, r, _, _ = _tiny("bf16")
    f1 = m.forward_feats(x)
    f2 = m.forward_feats(x.flip(0))
    with pytest.raises(vob.VitocmError, match="overwritten"):
        (f1 * r).sum().backward()
    (f2 * r).sum().backward()                      # the latest forward still has its activations


def test_mim_step_after_encoder_backward_on_the_same_engine():
    """An encoder backward binds its own gradient buffers; the next MIM backward must again accumulate into MIM's flat buffer and
    match the reference's golden step (tests/test_gpu_train.py's bars)."""
    g = load_golden("mim_train_tiny.npz")
    cfg_init = VO.ViTConfig(embed_dim=128, depth=2, num_heads=2, patch_size=8, img_size=224)
    sd = VO.randomize_affine(VO.init_state_dict(cfg_init, seed=11, mim=True), seed=12)
    enc = vob.VisionTransformerForSimMIM(patch_size=8, embed_dim=128, depth=2, num_heads=2, mlp_ratio=4, img_size=[32], qkv_bias=True,
                                         norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), precision="bf16")
    enc.load_state_dict(sd, strict=True)
    mim = vob.MIM(encoder=enc, encoder_stride=8)
    mim.decoder[0].weight.data.copy_(torch.from_numpy(g["dec_w"]))
    mim.decoder[0].bias.data.copy_(torch.from_numpy(g["dec_b"]))
    mim = mim.cuda().train()
    x, mask = torch.from_numpy(g["step0/x"]).cuda(), torch.from_numpy(g["step0/mask"]).cuda()
    for _ in range(2):
        mim.zero_grad(set_to_none=True)
        loss, _, _ = mim(x, mask)
        loss.sum().backward()
        mim.zero_grad(set_to_none=True)
        mim.encoder.forward_feats(x).square().sum().backward()
        assert mim.encoder.blocks[0].attn.qkv.weight.grad is not None
    mim.zero_grad(set_to_none=True)
    loss, _, _ = mim(x, mask)
    loss.sum().backward()
    num = den = 0.0
    worst = 0.0
    for n, p in mim.named_parameters():
        ref = g[f"step0/grad/{n[len('encoder.'):] if n.startswith('encoder.') else n}"]
        f = p.grad.detach().reshape(-1)
        got = (f if p.dim() <= 1 or f.numel() <= 4096 else f[::7]).cpu().numpy()
        d = got - ref
        worst = max(worst, float(np.abs(d).max() / max(np.abs(ref).max(), 1e-6)))
        num += float((d.astype(np.float64) ** 2).sum())
        den += float((ref.astype(np.float64) ** 2).sum())
    assert (num / den) ** 0.5 <= GRAD_TOL_GLOBAL and worst <= GRAD_TOL_TENSOR, ((num / den) ** 0.5, worst)


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_adamw_fine_tuning_lowers_the_loss_and_inference_tracks_the_oracle(precision):
    m, x, _, cfg, _ = _tiny(precision)
    head = torch.nn.Linear(cfg.embed_dim, N_CLASSES).cuda()
    labels = torch.arange(x.shape[0], device="cuda") % N_CLASSES
    opt = torch.optim.AdamW(list(m.parameters()) + list(head.parameters()), lr=1e-3, weight_decay=0.05)
    losses = []
    for _ in range(5):
        opt.zero_grad()
        loss = F.cross_entropy(head(m(x)), labels)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m.parameters(), 5.0)
        opt.step()
        losses.append(loss.item())
    assert losses[-1] < losses[0], losses
    m.eval()
    with torch.no_grad():
        got = m.forward_feats(x)
    sd = {k: v.detach().double().cpu() for k, v in m.state_dict().items()}
    ref = VO.forward_feats(sd, cfg, x.double().cpu())
    err = float((got.double().cpu() - ref).abs().max() / ref.abs().max())
    print(f"{precision}: losses {losses}; forward_feats after 5 steps off by {err:.3e} of the largest entry")
    assert err <= 2e-2


def test_encoder_backward_leaves_no_gradient_binding_behind():
    """The gradient buffers of an encoder backward are bound for that call only: a MIM step on an encoder without a qkv bias (MIM has
    no gradient buffer for it) is refused afterwards exactly as before, instead of accumulating into a freed buffer."""
    enc = vob.VisionTransformerForSimMIM(patch_size=8, embed_dim=128, depth=2, num_heads=2, mlp_ratio=4, img_size=[32], qkv_bias=False,
                                         norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), precision="bf16")
    mim = vob.MIM(encoder=enc, encoder_stride=8).cuda().train()
    x = torch.rand(2, 3, 32, 32, device="cuda")
    mask = torch.zeros(2, 4, 4, dtype=torch.int64, device="cuda")
    mask[:, :2] = 1
    enc.forward_feats(x).square().sum().backward()
    assert enc.blocks[0].attn.qkv.weight.grad is not None
    mim.zero_grad(set_to_none=True)
    loss, _, _ = mim(x, mask)
    with pytest.raises(vob.VitocmError, match="no bound gradient buffer"):
        loss.sum().backward()
