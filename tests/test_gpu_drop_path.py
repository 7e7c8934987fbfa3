"""GPU (B200): stochastic depth in the training kernels.

- Kernel level: the residual GEMM epilogue with a per-row scale (vitocm_gemm_resid_scaled) on single-CTA, B-resident and CTA-pair
  tiles, and the LayerNorm backward with a per-row scale (vitocm_layernorm_bwd_scaled) for every NV instantiation, at training launch
  sizes (M = 32 * 785 rows, samples of 785 rows whose boundaries fall mid-tile), NaN-guarded, against float64 / fp32 statements.
- Identity: all-ones scales give the plain forward's outputs bit for bit and its gradients up to the run-to-run order of the fp32
  atomics; a model with drop_path_rate > 0 in eval() gives bitwise what a rate-0 model gives.
- Oracle: explicit masks on the fine-tuning cases of tests/encoder_grad_cases.py and on a MIM step, against float64 autograd of a
  functional forward that scales the two branch adds of every block.
- Structure and RNG: a sample dropped everywhere gets norm(x_0); one seed gives the reference's masks."""
import math
from contextlib import contextmanager
from functools import partial

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import vitocm_b200 as vob
from encoder_grad_cases import CASES, inputs as _inputs, loss as _loss
from gpu_util import gemm, make_engine
from oracle import vit_oracle as VO
from vitocm_b200._lib import check, cur_stream, ptr

pytestmark = pytest.mark.gpu

GRAD_TOL_GLOBAL = 3e-2      # the bars of tests/test_gpu_encoder_grad.py
GRAD_TOL_TENSOR = 2e-1
EPS24 = 2.0 ** -24
DT = {"bf16": torch.bfloat16, "fp16": torch.float16}
FP16 = 2
PAD = 64
TOKENS = 785                 # 224^2 at patch 8: one sample's rows
M_TRAIN = 32 * TOKENS


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


@pytest.fixture(scope="module")
def engines():
    lib = vob._lib.load_library()
    e = {"bf16": make_engine(precision=0), "fp16": make_engine(precision=FP16)}
    yield e
    for h in e.values():
        lib.vitocm_destroy(h)


def _rand(shape, seed, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(shape, generator=g, device="cuda") * scale


def _sample_scales(n, seed):
    """per-sample scales cycling through drop, keep at 1 / 0.8, identity, and a large value; then shuffled"""
    vals = torch.tensor([0.0, 1.0 / 0.8, 1.0, 2.5], device="cuda")
    g = torch.Generator(device="cuda").manual_seed(seed)
    return vals[torch.arange(n, device="cuda") % 4][torch.randperm(n, generator=g, device="cuda")].contiguous()


def _rows(s, M, rps):
    return s[torch.arange(M, device="cuda") // rps][:, None]


# ------------------------------------------------------------------------------------------------------------ GEMM epilogue
# (M, N, K, path run_gemm takes on 148 SMs): proj of the training step (K = 384: B-resident, BN 128), fc2 (K = 1536: CTA pairs,
# BN 192), and K = 512 (single CTA, BN 128 / 64)
GEMM_PATHS = [(M_TRAIN, 384, 384, "resident-bn128"), (M_TRAIN, 384, 1536, "pair-bn192"), (M_TRAIN, 384, 512, "single-bn128"),
              (M_TRAIN, 128, 512, "single-bn64"), (3 * TOKENS + 5, 384, 384, "resident-ragged")]


def _resid_scaled(eng, A, W, b, X, ldx, M, N, K, s, rps):
    lib = vob._lib.load_library()
    check(lib.vitocm_gemm_resid_scaled(eng, ptr(A), A.stride(0), ptr(W), W.stride(0), M, N, K, ptr(b), ptr(X), ldx, ptr(s), rps,
                                       cur_stream()))
    torch.cuda.synchronize()


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("M,N,K,path", GEMM_PATHS, ids=[p[3] for p in GEMM_PATHS])
def test_gemm_residual_row_scale(engines, prec, M, N, K, path):
    """X += (A W^T + b) * s[row / 785].  With X = 0 the epilogue's fp32 values v come back exactly (checked against float64);
    the scaled call must then give fp32(X0 + fp32(v s)) bit for bit, and a NULL scale the existing epilogue's stores bit for bit.
    Pad rows and pad columns of X are NaN and must stay NaN."""
    eng, dt = engines[prec], DT[prec]
    A = _rand((M, K), 501).to(dt)
    W = _rand((N, K), 502, 1.0 / math.sqrt(K)).to(dt)
    b = _rand((N,), 503, 0.5)
    n_s = (M + TOKENS - 1) // TOKENS
    s = _sample_scales(n_s, 504)
    ldx = N + 64
    X0 = _rand((M, N), 505, 2.0)

    def run(x0, scale, plain=False):
        X = torch.full((M + PAD, ldx), float("nan"), device="cuda")
        X[:M, :N] = x0
        if plain:
            gemm(eng, A, W, M, N, K, 0, 2, b, X, ldx)
        else:
            _resid_scaled(eng, A, W, b, X, ldx, M, N, K, scale, TOKENS)
        assert torch.isnan(X[M:]).all() and torch.isnan(X[:M, N:]).all(), "a pad element was written"
        return X[:M, :N]

    zeros = torch.zeros(M, N, device="cuda")
    v = run(zeros, None, plain=True)
    ref = A.double() @ W.double().T + b.double()
    bound = (K + 2) * EPS24 * (A.double().abs() @ W.double().abs().T + b.double().abs())
    assert ((v.double() - ref).abs() <= bound).all(), "epilogue values off the float64 product"
    assert torch.equal(run(zeros, None), v)
    assert torch.equal(run(X0, None), run(X0, None, plain=True)), "NULL scale must store what epilogue 2 stores"
    sr = _rows(s, M, TOKENS)
    assert torch.equal(run(zeros, s), v * sr)
    got = run(X0, s)
    assert torch.equal(got, X0 + v * sr), "scaled residual add is not fp32(X0 + fp32(v s))"
    dropped = (sr == 0).expand(M, N)
    assert torch.equal(got[dropped], X0[dropped])


def test_gemm_row_scale_needs_rows_per_scale(engines):
    lib = vob._lib.load_library()
    A = torch.zeros(128, 64, device="cuda", dtype=torch.bfloat16)
    s = torch.ones(1, device="cuda")
    out = torch.zeros(128, 64, device="cuda")
    rc = lib.vitocm_gemm_resid_scaled(engines["bf16"], ptr(A), 64, ptr(A[:64]), 64, 128, 64, 64, None, ptr(out), 64, ptr(s), 0,
                                      cur_stream())
    assert rc != 0, "rows_per_scale 0 must be refused"


# ------------------------------------------------------------------------------------------------------------ LayerNorm backward
def _ln_call(eng, fn, X, dy, gamma, dX, dXb, sums, M, D, lscale, s=None, rps=1):
    lib = vob._lib.load_library()
    args = [eng, ptr(X), ptr(dy), D, ptr(gamma), ptr(dX), ptr(dXb), ptr(sums[0]), ptr(sums[1]), ptr(sums[2]), 1, M, D, ptr(lscale)]
    if fn == "scaled":
        check(lib.vitocm_layernorm_bwd_scaled(*args, ptr(s), rps, cur_stream()))
    else:
        check(lib.vitocm_layernorm_bwd(*args, cur_stream()))
    torch.cuda.synchronize()


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("D", [128, 384, 768, 256])
@pytest.mark.parametrize("M,rps", [(M_TRAIN, TOKENS), (1000, 7)])
def test_layernorm_backward_row_scale(engines, prec, D, M, rps):
    """NV = 1, 3, 6 and the generic path: dX (fp32) is that of vitocm_layernorm_bwd bit for bit; dXb is the 16-bit rounding of
    fp32(s dX) bit for bit; dbias_out is the column sums of s dX (float64, fp32-atomics bound); dgamma / dbeta are unscaled.  NULL
    gives vitocm_layernorm_bwd's dX and dXb bit for bit and its sums up to the order of the atomics."""
    eng, dt = engines[prec], DT[prec]
    X = _rand((M, D), 600 + D, 0.7) + _rand((M, 1), 601, 3.0)
    gamma = _rand((D,), 602) * 0.1 + 1.0
    dy = _rand((M, D), 603, 0.5).to(dt)
    dX_in = _rand((M, D), 604, 2.0)
    lscale = torch.ones(2, device="cuda") if prec == "fp16" else None
    n_s = (M + rps - 1) // rps
    s = _sample_scales(n_s, 605)

    def run(fn, scale=None):
        dX = dX_in.clone()
        dXb = torch.full((M + PAD, D), float("nan"), device="cuda", dtype=dt)
        sums = tuple(torch.zeros(D, device="cuda") for _ in range(3))
        _ln_call(eng, fn, X, dy, gamma, dX, dXb, sums, M, D, lscale, scale, rps)
        assert torch.isnan(dXb[M:].float()).all(), "a pad row of dXb was written"
        return dX, dXb[:M], sums

    # fp32 atomics: each column sum is within n_add 2^-24 sum |terms| of its exact value, in whatever order the atomics land
    grid = min((M + 63) // 64, 296)
    n_add = (M + grid * 8 - 1) // (grid * 8) + 8 + grid + 2
    X64 = X.double()
    xhat = (X64 - X64.mean(1, keepdim=True)) / torch.sqrt(X64.var(1, unbiased=False, keepdim=True) + 1e-6)
    abs_terms = [(dy.double() * xhat).abs().sum(0), dy.double().abs().sum(0)]

    def close(a, b, terms, what):
        assert ((a.double() - b.double()).abs() <= 2 * n_add * EPS24 * terms + 1e-30).all(), what

    dX1, dXb1, sums1 = run("plain")
    dX2, dXb2, sums2 = run("scaled")
    assert torch.equal(dX2, dX1) and torch.equal(dXb2.view(torch.int16), dXb1.view(torch.int16))
    abs_terms.append(dX1.double().abs().sum(0))
    for a, b, t, what in zip(sums2, sums1, abs_terms, ("dgamma", "dbeta", "dbias_out")):
        close(a, b, t, f"NULL scale: {what}")
    dX3, dXb3, sums3 = run("scaled", s)
    assert torch.equal(dX3, dX1), "the identity path must stay unscaled"
    sdx = dX1 * _rows(s, M, rps)
    want = sdx.clamp(-65504, 65504).half() if prec == "fp16" else sdx.to(torch.bfloat16)
    assert torch.equal(dXb3.view(torch.int16), want.view(torch.int16)), "dXb is not the 16-bit rounding of s dX"
    close(sums3[0], sums1[0], abs_terms[0], "dgamma must be unscaled")
    close(sums3[1], sums1[1], abs_terms[1], "dbeta must be unscaled")
    ref = sdx.double().sum(0)
    bound = n_add * EPS24 * sdx.double().abs().sum(0) + 1e-30
    assert ((sums3[2].double() - ref).abs() <= bound).all(), "dbias_out is not the column sums of s dX"


# ------------------------------------------------------------------------------------------------------------ model level
@contextmanager
def forced_scales(enc, scales):
    """The training forwards of ``enc`` use ``scales`` [depth, 2, B] instead of drawing them."""
    enc._branch_scales = lambda B, dev: scales
    try:
        yield
    finally:
        del enc._branch_scales


def _model(cfg, sd, precision, rate=0.0):
    m = vob.VisionTransformer(img_size=[cfg.img_size], patch_size=cfg.patch_size, embed_dim=cfg.embed_dim, depth=cfg.depth,
                              num_heads=cfg.num_heads, mlp_ratio=cfg.mlp_ratio, qkv_bias=True,
                              norm_layer=partial(torch.nn.LayerNorm, eps=cfg.eps), precision=precision, drop_path_rate=rate)
    m.load_state_dict(sd, strict=True)
    return m.cuda().train()


def explicit_masks(depth, B, seed, keep=0.75):
    """[depth, 2, B]: sample 0 dropped in every branch, sample 1 kept in every branch, the others drawn per branch"""
    g = torch.Generator().manual_seed(seed)
    r = (torch.rand(depth, 2, B, generator=g) < keep).float()
    r[:, :, 0] = 0.0
    r[:, :, 1] = 1.0
    return (r / keep).cuda()


def oracle_feats_dp(sd, cfg, x, n, s):
    """get_intermediate_layers over oracle/vit_oracle.py's pieces with block i's two residual adds scaled by s[i, 0] / s[i, 1]"""
    t = VO.prepare_tokens(sd, cfg, x)
    outs = []
    for i in range(cfg.depth):
        pre = f"blocks.{i}."
        y, _, _ = VO.attention(sd, cfg, i, VO._ln(t, sd[pre + "norm1.weight"], sd[pre + "norm1.bias"], cfg.eps))
        t = t + y * s[i, 0][:, None, None]
        t = t + VO.mlp(sd, cfg, i, VO._ln(t, sd[pre + "norm2.weight"], sd[pre + "norm2.bias"], cfg.eps)) * s[i, 1][:, None, None]
        if cfg.depth - i <= n:
            outs.append(VO._ln(t, sd["norm.weight"], sd["norm.bias"], cfg.eps))
    return outs


def _grad_vector(m, xc):
    return torch.cat([p.grad.reshape(-1) for p in m.parameters()] + [xc.grad.reshape(-1)])


def _encoder_pass(m, x, r):
    """forward + backward of get_intermediate_layers(n=2) (the injected-feature path) -> (features, gradient vector)"""
    m.zero_grad(set_to_none=True)
    xc = x.clone().requires_grad_(True)
    feats = m.get_intermediate_layers(xc, n=2)
    sum((f * rr).sum() for f, rr in zip(feats, r)).backward()
    return [f.detach().clone() for f in feats], _grad_vector(m, xc)


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("case", ["tiny-48x64", "reference-encoder"])
def test_encoder_all_ones_scales_are_the_plain_step(precision, case):
    """Single-CTA tiles (tiny) and B-resident / CTA-pair tiles (reference encoder, batch 8): feats bitwise; every gradient, dpos
    (pos_embed's gradient) and dx within the spread of two plain runs."""
    cfg, H, W, B = CASES[case]
    sd = VO.randomize_affine(VO.init_state_dict(cfg, seed=41), seed=42)
    x, _ = _inputs(cfg, H, W, B, seed=43)
    x = x.cuda()
    N = (H // cfg.patch_size) * (W // cfg.patch_size) + 1
    r = [_rand((B, N, cfg.embed_dim), 44 + k) for k in range(2)]
    m = _model(cfg, sd, precision)
    f0, g0 = _encoder_pass(m, x, r)
    _, g0b = _encoder_pass(m, x, r)
    spread = (g0b - g0).abs().max().item()
    with forced_scales(m, torch.ones(cfg.depth, 2, B, device="cuda")):
        f1, g1 = _encoder_pass(m, x, r)
    for a, b in zip(f1, f0):
        assert torch.equal(a, b)
    diff = (g1 - g0).abs().max().item()
    assert diff <= 2 * spread + 1e-7 * g0.abs().max().item(), (diff, spread)


def _mim_setup(precision, rate=0.0, seed=11):
    cfg_init = VO.ViTConfig(embed_dim=128, depth=2, num_heads=2, patch_size=8, img_size=224)
    cfg = VO.ViTConfig(embed_dim=128, depth=2, num_heads=2, patch_size=8, img_size=32)
    sd = VO.randomize_affine(VO.init_state_dict(cfg_init, seed=seed, mim=True), seed=seed + 1)
    gd = torch.Generator().manual_seed(seed + 2)
    dec_w, dec_b = torch.randn(192, 128, 1, 1, generator=gd) * 0.05, torch.randn(192, generator=gd) * 0.05
    enc = vob.VisionTransformerForSimMIM(patch_size=8, embed_dim=128, depth=2, num_heads=2, mlp_ratio=4, img_size=[32], qkv_bias=True,
                                         norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), precision=precision, drop_path_rate=rate)
    enc.load_state_dict(sd, strict=True)
    mim = vob.MIM(encoder=enc, encoder_stride=8)
    mim.decoder[0].weight.data.copy_(dec_w)
    mim.decoder[0].bias.data.copy_(dec_b)
    mim = mim.cuda().train()
    B = 6
    x = VO.synthetic_tile(32, seed=77, batch=B)
    rs = np.random.RandomState(3)
    masks = torch.from_numpy(np.stack([VO.mask_generator(rs, 32, 16, 8, 0.5) for _ in range(B)]))
    params = dict(sd)
    params["decoder.0.weight"], params["decoder.0.bias"] = dec_w, dec_b
    return mim, cfg, params, x, masks


def _mim_pass(mim, x, mask):
    mim.zero_grad(set_to_none=True)
    loss, x_rec, _ = mim(x.cuda(), mask.cuda())
    loss.sum().backward()
    return loss.detach().clone(), x_rec.detach().clone(), torch.cat([p.grad.reshape(-1) for p in mim.parameters()])


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_mim_all_ones_scales_are_the_plain_step(precision):
    mim, cfg, _, x, masks = _mim_setup(precision)
    l0, xr0, g0 = _mim_pass(mim, x, masks)
    _, _, g0b = _mim_pass(mim, x, masks)
    spread = (g0b - g0).abs().max().item()
    with forced_scales(mim.encoder, torch.ones(cfg.depth, 2, x.shape[0], device="cuda")):
        l1, xr1, g1 = _mim_pass(mim, x, masks)
    assert torch.equal(xr1, xr0)
    assert abs(l1.item() - l0.item()) <= 1e-6 * abs(l0.item())       # fp64 atomics of the loss sums
    assert (g1 - g0).abs().max().item() <= 2 * spread + 1e-7 * g0.abs().max().item()


def test_eval_mode_ignores_the_rate():
    """drop path is the identity in eval(): a rate-0.3 model runs exactly the rate-0 model's inference path"""
    cfg, H, W, B = CASES["tiny-48x64"]
    sd = VO.randomize_affine(VO.init_state_dict(cfg, seed=51), seed=52)
    x, _ = _inputs(cfg, H, W, B, seed=53)
    x = x.cuda()
    m0, m3 = _model(cfg, sd, "bf16").eval(), _model(cfg, sd, "bf16", rate=0.3).eval()
    assert torch.equal(m3.cls_attention_rows(x), m0.cls_attention_rows(x))
    assert torch.equal(m3.forward_feats(x), m0.forward_feats(x))
    mim0, _, _, xm, masks = _mim_setup("bf16")
    mim3, _, _, _, _ = _mim_setup("bf16", rate=0.3)
    mim0.eval(); mim3.eval()
    with torch.no_grad():
        a, ra, _ = mim0(xm.cuda(), masks.cuda())
        b, rb, _ = mim3(xm.cuda(), masks.cuda())
    assert torch.equal(ra, rb)
    assert abs(a.item() - b.item()) <= 1e-12 * abs(a.item())


def _errors(model, ref, x_grad, ref_dx):
    num = den = 0.0
    worst = (0.0, "")
    for n, p in model.named_parameters():
        r = ref[n]
        d = (p.grad.double() - r).reshape(-1)
        num += float(d.pow(2).sum())
        den += float(r.pow(2).sum())
        worst = max(worst, (float(d.abs().max() / r.abs().max().clamp_min(1e-30)), n))
    dx_rel = float((x_grad.double() - ref_dx).norm() / ref_dx.norm())
    dx_max = float((x_grad.double() - ref_dx).abs().max() / ref_dx.abs().max())
    return (num / den) ** 0.5, worst, dx_rel, dx_max


@pytest.mark.parametrize("upstream", ["head", "feats", "intermediate"])
@pytest.mark.parametrize("case", list(CASES))
def test_gradients_match_float64_oracle_with_explicit_masks(case, upstream):
    cfg, H, W, B = CASES[case]
    sd = VO.randomize_affine(VO.init_state_dict(cfg, seed=21), seed=22)
    x, u = _inputs(cfg, H, W, B, seed=23)
    s = explicit_masks(cfg.depth, B, seed=24)
    s64 = s.double()
    leaves = {k: v.detach().double().cuda().requires_grad_(True) for k, v in sd.items()}
    xd = x.double().cuda().requires_grad_(True)
    feats = lambda n: oracle_feats_dp(leaves, cfg, xd, n, s64)   # noqa: E731
    _loss(upstream, lambda: feats(1)[0], lambda: feats(1)[0][:, 0], lambda: feats(4), u, torch.float64, "cuda").backward()
    ref, ref_dx = {k: v.grad for k, v in leaves.items()}, xd.grad
    for precision in ("bf16", "fp16"):
        m = _model(cfg, sd, precision, rate=0.1)
        xc = x.cuda().requires_grad_(True)
        with forced_scales(m, s):
            loss = _loss(upstream, lambda: m.forward_feats(xc), lambda: m(xc), lambda: m.get_intermediate_layers(xc, n=4), u,
                         torch.float32, "cuda")
            loss.backward()
        g, worst, dx_rel, dx_max = _errors(m, ref, xc.grad, ref_dx)
        print(f"{case} {upstream} {precision}: global {g:.3e}, worst tensor {worst[0]:.3e} ({worst[1]}), dx {dx_rel:.3e} / {dx_max:.3e}")
        assert g <= GRAD_TOL_GLOBAL, (precision, g)
        assert worst[0] <= GRAD_TOL_TENSOR, (precision, worst)
        assert dx_rel <= GRAD_TOL_GLOBAL and dx_max <= GRAD_TOL_TENSOR, (precision, dx_rel, dx_max)
        del m


def _mim_oracle(params, cfg, x, mask, s64):
    """oracle/vit_oracle.py's MIM forward (simmim_encoder + decoder + masked L1) with scaled branch adds -> (loss, {key: grad})"""
    leaves = {k: v.detach().double().cuda().requires_grad_(True) for k, v in params.items()}
    sd = {k: v for k, v in leaves.items() if not k.startswith("decoder.")}
    xd, md = x.double().cuda(), mask.cuda()
    t = VO.patch_embed(sd, cfg, xd)
    B, L, _ = t.shape
    w = md.flatten(1).unsqueeze(-1).type_as(t)
    t = t * (1 - w) + sd["mask_token"].expand(B, L, -1) * w
    t = torch.cat((sd["cls_token"].expand(B, -1, -1), t), dim=1)
    t = t + VO.interpolate_pos_encoding(sd, cfg, L, cfg.img_size, cfg.img_size)
    for i in range(cfg.depth):
        pre = f"blocks.{i}."
        y, _, _ = VO.attention(sd, cfg, i, VO._ln(t, sd[pre + "norm1.weight"], sd[pre + "norm1.bias"], cfg.eps))
        t = t + y * s64[i, 0][:, None, None]
        t = t + VO.mlp(sd, cfg, i, VO._ln(t, sd[pre + "norm2.weight"], sd[pre + "norm2.bias"], cfg.eps)) * s64[i, 1][:, None, None]
    t = VO._ln(t, sd["norm.weight"], sd["norm.bias"], cfg.eps)[:, 1:]
    Hh = int(L ** 0.5)
    z = t.permute(0, 2, 1).reshape(B, -1, Hh, Hh)
    x_rec = F.pixel_shuffle(F.conv2d(z, leaves["decoder.0.weight"], leaves["decoder.0.bias"]), cfg.patch_size)
    m = md.repeat_interleave(cfg.patch_size, 1).repeat_interleave(cfg.patch_size, 2).unsqueeze(1).double()
    loss = (F.l1_loss(xd, x_rec, reduction="none") * m).sum() / (m.sum() + 1e-5) / cfg.in_chans
    loss.backward()
    return loss.detach(), {k: v.grad for k, v in leaves.items()}


def _mim_errors(mim, ref):
    num = den = 0.0
    worst = 0.0
    for n, p in mim.named_parameters():
        r = ref[n[len("encoder."):] if n.startswith("encoder.") else n]
        d = (p.grad.double() - r).reshape(-1)
        num += float(d.pow(2).sum())
        den += float(r.pow(2).sum())
        worst = max(worst, float(d.abs().max() / r.abs().max().clamp_min(1e-30)))
    return (num / den) ** 0.5, worst


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_mim_step_matches_float64_oracle_with_explicit_masks(precision):
    mim, cfg, params, x, masks = _mim_setup(precision, rate=0.1)
    s = explicit_masks(cfg.depth, x.shape[0], seed=61)
    ref_loss, ref = _mim_oracle(params, cfg, x, masks, s.double())
    with forced_scales(mim.encoder, s):
        loss, _, _ = _mim_pass(mim, x, masks)
    g, worst = _mim_errors(mim, ref)
    print(f"MIM {precision}: loss {loss.item():.6f} vs {ref_loss.item():.6f}, global {g:.3e}, worst tensor {worst:.3e}")
    assert abs(loss.item() - ref_loss.item()) <= 2e-2 * abs(ref_loss.item())
    assert g <= GRAD_TOL_GLOBAL and worst <= GRAD_TOL_TENSOR, (g, worst)


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_mim_backward_uses_its_own_forwards_masks_when_workspaces_interleave(precision):
    """MIM forward with masks -> an encoder forward + backward without drop path on the same engine -> the MIM backward: its
    gradients still follow the MIM forward's masks (the oracle's bars)."""
    mim, cfg, params, x, masks = _mim_setup(precision, rate=0.1)
    s = explicit_masks(cfg.depth, x.shape[0], seed=62)
    _, ref = _mim_oracle(params, cfg, x, masks, s.double())
    mim.zero_grad(set_to_none=True)
    with forced_scales(mim.encoder, s):
        loss, _, _ = mim(x.cuda(), masks.cuda())
    enc = mim.encoder
    with forced_scales(enc, None):
        enc.forward_feats(x.cuda()).square().sum().backward()
    mim.zero_grad(set_to_none=True)
    loss.sum().backward()
    g, worst = _mim_errors(mim, ref)
    assert g <= GRAD_TOL_GLOBAL and worst <= GRAD_TOL_TENSOR, (g, worst)


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_sample_dropped_everywhere_is_the_normalised_embedding(precision):
    """x_L = x_0 for a sample whose every branch is dropped, so its feature is norm(x_0) up to fp32 LayerNorm rounding; under
    no_grad in training mode too."""
    cfg, H, W, B = CASES["tiny-48x64"]
    sd = VO.randomize_affine(VO.init_state_dict(cfg, seed=71), seed=72)
    x, _ = _inputs(cfg, H, W, B, seed=73)
    x = x.cuda()
    m = _model(cfg, sd, precision, rate=0.2)
    s = explicit_masks(cfg.depth, B, seed=74)
    with forced_scales(m, s), torch.no_grad():
        feats = m.forward_feats(x)
    assert feats.grad_fn is None
    x0 = m.prepare_tokens(x)
    want = F.layer_norm(x0[0], (cfg.embed_dim,), m.norm.weight.detach(), m.norm.bias.detach(), cfg.eps)
    assert (feats[0] - want).abs().max().item() <= 5e-5 * max(1.0, want.abs().max().item())
    assert (feats[1] - want).abs().max().item() > 1e-2        # a kept sample does go through the blocks


def test_one_seed_gives_the_reference_masks_and_the_oracle_loss():
    """Under torch.manual_seed on the device the module draws what DINO's drop_path calls draw (block by block, attn then mlp, no
    draw for block 0), and its loss matches the float64 oracle run with those masks."""
    cfg, H, W, _ = CASES["tiny-48x64"]
    B = 16
    sd = VO.randomize_affine(VO.init_state_dict(cfg, seed=81), seed=82)
    x, u = _inputs(cfg, H, W, B, seed=83)
    m = _model(cfg, sd, "bf16", rate=0.5)
    drawn = []
    orig = m._branch_scales
    m._branch_scales = lambda b, dev: drawn.append(orig(b, dev)) or drawn[-1]
    torch.manual_seed(1234)
    feats = m.forward_feats(x.cuda())
    loss = (feats * u["r_feats"].cuda()).sum()
    del m._branch_scales

    torch.manual_seed(1234)
    ref = torch.ones(cfg.depth, 2, B, device="cuda")
    for l, p in enumerate(v.item() for v in torch.linspace(0, 0.5, cfg.depth)):
        for k in range(2):
            if p > 0:                      # DropPath(p) for p > 0, nn.Identity otherwise (vit.py:101)
                keep = 1 - p
                r = torch.floor(keep + torch.rand((B, 1, 1), dtype=torch.float32, device="cuda"))
                ref[l, k] = (torch.ones(B, 1, 1, device="cuda").div(keep) * r).reshape(B)
    assert len(drawn) == 1 and torch.equal(drawn[0], ref)
    assert (ref == 0).any() and (ref > 1).any()
    sd64 = {k: v.double().cuda() for k, v in sd.items()}
    with torch.no_grad():
        f64 = oracle_feats_dp(sd64, cfg, x.double().cuda(), 1, ref.double())[0]
        ref_loss = (f64 * u["r_feats"].cuda().double()).sum().item()
    assert float((feats.double() - f64).norm() / f64.norm()) <= GRAD_TOL_GLOBAL
    assert abs(loss.item() - ref_loss) <= GRAD_TOL_GLOBAL * (f64 * u["r_feats"].cuda().double()).abs().sum().item()
