"""GPU (B200): each hand-written kernel against a plain fp32 torch statement of the same op,
called through the C ABI."""
import math

import pytest
import torch

import block_half_oracle as BO
import vitocm_b200 as vob
from gpu_util import attention, attention_reference, gemm, make_engine, split_bf16
from vitocm_b200._lib import check, cur_stream, ptr

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


@pytest.fixture(scope="module")
def engine():
    return make_engine()


def _rand(shape, seed, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(shape, generator=g, device="cuda") * scale


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (300, 256, 128), (785, 1152, 384), (1570, 1536, 384),
                                   (785, 384, 1536), (200, 192, 192), (77, 64, 64), (2355, 320, 384)])
def test_gemm_bias_bf16(engine, M, N, K):
    A = _rand((M, K), 1).to(torch.bfloat16)
    B = _rand((N, K), 2, 0.05).to(torch.bfloat16)
    bias = _rand((N,), 3, 0.1)
    out = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
    gemm(engine, A, B, M, N, K, 0, 0, bias, out, N)
    ref = A.float() @ B.float().T + bias
    err = (out.float() - ref).abs().max().item()
    assert err <= 2e-2 * ref.abs().max().item() + 1e-3, err
    assert torch.isfinite(out.float()).all()


def test_gemm_gelu_epilogue(engine):
    M, N, K = 785, 1536, 384
    A = _rand((M, K), 4).to(torch.bfloat16)
    B = _rand((N, K), 5, 0.08).to(torch.bfloat16)
    bias = _rand((N,), 6, 0.2)
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    gemm(engine, A, B, M, N, K, 0, 1, bias, out, N)
    ref = torch.nn.functional.gelu(A.float() @ B.float().T + bias)
    assert (out.float() - ref).abs().max().item() <= 1e-2 * ref.abs().max().item() + 1e-3


def test_gemm_residual_and_f32_epilogues(engine):
    M, N, K = 1000, 384, 1536
    A = _rand((M, K), 7).to(torch.bfloat16)
    B = _rand((N, K), 8, 0.03).to(torch.bfloat16)
    bias = _rand((N,), 9, 0.1)
    resid = _rand((M, N), 10)
    ref = resid + A.float() @ B.float().T + bias
    x = resid.clone()
    gemm(engine, A, B, M, N, K, 0, 2, bias, x, N)
    assert (x - ref).abs().max().item() <= 2e-4 * ref.abs().max().item()
    y = torch.empty(M, N, device="cuda")
    gemm(engine, A, B, M, N, K, 0, 3, bias, y, N)
    assert (y - (ref - resid)).abs().max().item() <= 2e-4 * ref.abs().max().item()


@pytest.mark.parametrize("M,N,K", [(1000, 384, 384), (3000, 768, 256), (25120, 384, 384), (130, 128, 64)])
def test_gemm_weight_panel_resident_epilogues(engine, M, N, K):
    """K <= 384 with single-bf16 operands takes the weight-panel-resident kernel (n-major contiguous tile ranges,
    panel reloads when a CTA crosses into the next column of tiles)."""
    A = _rand((M, K), 30).to(torch.bfloat16)
    B = _rand((N, K), 31, 0.05).to(torch.bfloat16)
    bias = _rand((N,), 32, 0.1)
    resid = _rand((M, N), 33)
    prod = A.float() @ B.float().T + bias
    x = resid.clone()
    gemm(engine, A, B, M, N, K, 0, 2, bias, x, N)
    assert (x - (resid + prod)).abs().max().item() <= 2e-4 * prod.abs().max().item() + 1e-5
    y = torch.full((M, N), float("nan"), device="cuda")
    gemm(engine, A, B, M, N, K, 0, 3, bias, y, N)
    assert (y - prod).abs().max().item() <= 2e-4 * prod.abs().max().item() + 1e-5
    z = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
    gemm(engine, A, B, M, N, K, 0, 1, bias, z, N)
    ref = torch.nn.functional.gelu(prod)
    assert (z.float() - ref).abs().max().item() <= 1e-2 * ref.abs().max().item() + 1e-3


@pytest.mark.parametrize("M,N,K", [(1000, 384, 384), (25120, 384, 1536), (300, 128, 128), (777, 768, 384), (500, 512, 64), (900, 256, 128)])
def test_gemm_fused_residual_layernorm(engine, M, N, K):
    """proj / fc2 epilogue with the next LayerNorm fused: a row spans N / BN CTAs of one cluster which exchange
    (mean, M2) partials through distributed shared memory."""
    lib = vob._lib.load_library()
    A = _rand((M, K), 40).to(torch.bfloat16)
    B = _rand((N, K), 41, 0.05).to(torch.bfloat16)
    bias = _rand((N,), 42, 0.1)
    resid = _rand((M, N), 43) + 0.3
    gamma, beta = _rand((N,), 44) * 0.1 + 1, _rand((N,), 45) * 0.1
    x = resid.clone()
    xn = torch.full((M, 2 * N), float("nan"), device="cuda", dtype=torch.bfloat16)
    check(lib.vitocm_gemm_ln(engine, ptr(A), A.stride(0), ptr(B), B.stride(0), M, N, K, ptr(bias), ptr(x), ptr(gamma), ptr(beta),
                             ptr(xn), xn.stride(0), cur_stream()))
    torch.cuda.synchronize()
    ref_x = resid + A.float() @ B.float().T + bias
    assert (x - ref_x).abs().max().item() <= 2e-4 * ref_x.abs().max().item() + 1e-5
    ref_n = torch.nn.functional.layer_norm(x, (N,), gamma, beta, 1e-6)          # LN of the kernel's own updated rows
    assert (xn[:, :N].float() - ref_n).abs().max().item() <= 2e-2
    assert torch.isnan(xn[:, N:].float()).all()                                   # lo half untouched


@pytest.mark.parametrize("M,N,K,epi", [(70000, 1152, 384, 0), (66000, 1536, 384, 1), (5000, 384, 1536, 2), (4100, 256, 1024, 3),
                                       (65537, 128, 64, 0)])
def test_gemm_cta_pair_mode(engine, M, N, K, epi):
    """Shapes that take the cta_group::2 kernel (CTA pairs on 256-row tiles, each CTA staging half of the B tile)."""
    A = _rand((M, K), 50).to(torch.bfloat16)
    B = _rand((N, K), 51, 0.05).to(torch.bfloat16)
    bias = _rand((N,), 52, 0.1)
    prod = A.float() @ B.float().T + bias
    if epi <= 1:
        out = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
        gemm(engine, A, B, M, N, K, 0, epi, bias, out, N)
        ref = torch.nn.functional.gelu(prod) if epi == 1 else prod
        assert (out.float() - ref).abs().max().item() <= 1e-2 * ref.abs().max().item() + 1e-3
    else:
        resid = _rand((M, N), 53)
        out = resid.clone() if epi == 2 else torch.full((M, N), float("nan"), device="cuda")
        gemm(engine, A, B, M, N, K, 0, epi, bias, out, N)
        ref = resid + prod if epi == 2 else prod
        assert (out - ref).abs().max().item() <= 2e-4 * ref.abs().max().item() + 1e-5


def test_gemm_split_precision_is_fp32_grade(engine):
    M, N, K = 785, 384, 384
    A32, B32 = _rand((M, K), 11), _rand((N, K), 12, 0.05)
    bias = _rand((N,), 13, 0.1)
    A, B = split_bf16(A32), split_bf16(B32)
    y = torch.empty(M, N, device="cuda")
    gemm(engine, A, B, M, N, K, 1, 3, bias, y, N)
    ref = (A32.double() @ B32.double().T + bias.double()).float()
    rel = ((y - ref).abs().max() / ref.abs().max()).item()
    assert rel < 2e-5, rel
    # split output: hi | lo reconstructs the fp32 value
    out = torch.empty(M, 2 * N, device="cuda", dtype=torch.bfloat16)
    gemm(engine, A, B, M, N, K, 1, 0, bias, out, 2 * N, 1, N)
    rec = out[:, :N].float() + out[:, N:].float()
    assert ((rec - ref).abs().max() / ref.abs().max()).item() < 5e-5


def test_layernorm(engine):
    lib = vob._lib.load_library()
    M, D = 1000, 128
    x = _rand((M, D), 14, 3.0) + 0.5
    g, b = _rand((D,), 15) * 0.1 + 1, _rand((D,), 16) * 0.1
    out = torch.empty(M, 2 * D, device="cuda", dtype=torch.bfloat16)
    check(lib.vitocm_layernorm(engine, ptr(x), ptr(g), ptr(b), ptr(out), 2 * D, 1, D, M, cur_stream()))
    torch.cuda.synchronize()
    ref = torch.nn.functional.layer_norm(x, (D,), g, b, 1e-6)
    assert (out[:, :D].float() - ref).abs().max().item() < 2e-2
    assert ((out[:, :D].float() + out[:, D:].float()) - ref).abs().max().item() < 1e-4


# ragged query tails: 17 / 129 / 150 / 785 pack four (image, head) pairs into one tile, 300 / 37 two, 65 / 200 none; 2, 6 and 10
# pairs leave the last group of a packed launch partly empty
@pytest.mark.parametrize("B,H,N", [(1, 2, 17), (2, 2, 65), (1, 2, 128), (1, 2, 129), (2, 2, 300), (1, 6, 785), (3, 2, 37), (5, 2, 150),
                                   (7, 2, 200), (4, 6, 785)])
@pytest.mark.parametrize("precision", [0, 1])
def test_attention(B, H, N, precision):
    eng = make_engine(embed_dim=64 * H, heads=H, precision=precision)
    D = 64 * H
    q, k, v = (_rand((B, H, N, 64), s, sc) for s, sc in ((20, 1.0), (21, 1.0), (22, 1.0)))
    parts = 2 if precision else 1
    # [B*N, 3D] layout with columns [3][H][64]
    qkv32 = torch.stack([q, k, v], 0).permute(1, 3, 0, 2, 4).reshape(B * N, 3 * D).contiguous()
    if precision:
        qkv = split_bf16(qkv32)
        qr = kr = vr = None
        src = qkv[:, :3 * D].float() + qkv[:, 3 * D:].float()
    else:
        qkv = qkv32.to(torch.bfloat16).contiguous()
        src = qkv.float()
    s5 = src.reshape(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
    ref = attention_reference(s5[0], s5[1], s5[2], 0.125).reshape(B * N, D)
    ctx = torch.full((B * N, D * parts), float("nan"), device="cuda", dtype=torch.bfloat16)
    attention(eng, qkv, B, N, ctx)
    got = ctx[:, :D].float() + (ctx[:, D:].float() if precision else 0)
    err = (got - ref).abs().max().item()
    tol = 3e-5 if precision else 2e-2
    assert err <= tol * max(1.0, ref.abs().max().item()), (err, ref.abs().max().item())
    vob._lib.load_library().vitocm_destroy(eng)


@pytest.mark.parametrize("gain", [6.0, 60.0])
def test_attention_rising_logits_rescale_and_redo(gain):
    """Logits that grow along the key axis: later KV blocks exceed the running row maximum by 2^8 (lazy rescale of
    O / l before the next block) and, at the larger gain, by more than 2^60 inside one block (the block is redone
    against the raised maximum instead of overflowing exp2)."""
    B, H, N, precision = 1, 2, 600, 0
    eng = make_engine(embed_dim=64 * H, heads=H, precision=precision)
    D = 64 * H
    q, k, v = (_rand((B, H, N, 64), s) for s in (60, 61, 62))
    ramp = torch.linspace(0.2, 1.0, N, device="cuda").view(1, 1, N, 1)
    k = k * ramp * gain                                  # |logit| grows with the key index
    qkv = torch.stack([q, k, v], 0).permute(1, 3, 0, 2, 4).reshape(B * N, 3 * D).to(torch.bfloat16).contiguous()
    s5 = qkv.float().reshape(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
    ref = attention_reference(s5[0], s5[1], s5[2], 0.125).reshape(B * N, D)
    ctx = torch.full((B * N, D), float("nan"), device="cuda", dtype=torch.bfloat16)
    attention(eng, qkv, B, N, ctx)
    assert torch.isfinite(ctx.float()).all()
    assert (ctx.float() - ref).abs().max().item() <= 3e-2 * max(1.0, ref.abs().max().item())
    vob._lib.load_library().vitocm_destroy(eng)


def test_launch_counter_counts():
    before = vob._lib.launch_count()
    eng = make_engine()
    A = torch.zeros(128, 64, device="cuda", dtype=torch.bfloat16)
    out = torch.empty(128, 64, device="cuda", dtype=torch.bfloat16)
    gemm(eng, A, A[:64].contiguous(), 128, 64, 64, 0, 0, None, out, 64)
    assert vob._lib.launch_count() == before + 1


def _mlp_reference(A, W1, b1, W2, b2, resid, dt):
    """fp32 statement of Mlp.forward + residual with the hidden activations rounded to the engine's 16-bit format (the fused
    kernel keeps them in shared memory in that format)."""
    hid = torch.nn.functional.gelu(A.float() @ W1.float().T + b1).to(dt).float()
    return resid + hid @ W2.float().T + b2


@pytest.mark.parametrize("M,D,Hd", [(785, 384, 1536), (256, 384, 1536), (130, 128, 512), (1, 128, 128), (5000, 384, 1536), (40000, 384, 1536),
                                    (257, 128, 256), (40000, 128, 384), (60000, 128, 128)])   # odd chunk counts: the epilogue groups swap per item
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_mlp_fused(M, D, Hd, precision):
    """fc1 + GELU + fc2 + residual in one kernel (CTA pairs, hidden chunks through TMEM and shared memory): ragged row tiles, one
    and many items per pair, both instantiated widths."""
    lib = vob._lib.load_library()
    eng = make_engine(precision=2 if precision == "fp16" else 0)
    dt = torch.float16 if precision == "fp16" else torch.bfloat16
    # strided rows like the workspace's XN [M][2D]; the unused half is NaN
    A2 = torch.cat([_rand((M, D), 60).to(dt), torch.full((M, D), float("nan"), device="cuda", dtype=dt)], dim=1).contiguous()
    A = A2[:, :D]
    W1 = _rand((Hd, D), 61, 0.06).to(dt)
    W2 = _rand((D, Hd), 62, 0.03).to(dt)
    b1, b2 = _rand((Hd,), 63, 0.2), _rand((D,), 64, 0.1)
    resid = _rand((M, D), 65)
    x = resid.clone()
    check(lib.vitocm_mlp_fused(eng, ptr(A2), A2.stride(0), ptr(W1), W1.stride(0), ptr(W2), W2.stride(0), M, D, Hd, ptr(b1), ptr(b2), ptr(x),
                               cur_stream()))
    torch.cuda.synchronize()
    ref = _mlp_reference(A, W1, b1, W2, b2, resid, dt)
    tol = 3e-3 if precision == "fp16" else 1.5e-2     # the GELU approximation and the fp32 summation order differ from torch's
    err = (x - ref).abs().max().item()
    assert err <= tol * (ref - resid).abs().max().item() + 1e-4, err
    # twice on the same residual stream = two blocks' worth of accumulation (reduce-add, not overwrite)
    check(lib.vitocm_mlp_fused(eng, ptr(A2), A2.stride(0), ptr(W1), W1.stride(0), ptr(W2), W2.stride(0), M, D, Hd, ptr(b1), ptr(b2), ptr(x),
                               cur_stream()))
    torch.cuda.synchronize()
    ref2 = ref + (ref - resid)
    assert (x - ref2).abs().max().item() <= 2 * tol * (ref - resid).abs().max().item() + 2e-4


def _tail_reference(ctx, Wp, bp, g2, be2, W1, b1, W2, b2, gn, ben, resid, dt, eps=1e-6):
    """fp32 statement of the second half of Block.forward with the two activations the kernel keeps in 16 bits (norm2's output and
    the hidden chunk) rounded to the engine's format."""
    x = resid + ctx.float() @ Wp.float().T + bp
    xn2 = torch.nn.functional.layer_norm(x, (x.shape[1],), g2, be2, eps).to(dt).float()
    hid = torch.nn.functional.gelu(xn2 @ W1.float().T + b1).to(dt).float()
    x = x + hid @ W2.float().T + b2
    xn = torch.nn.functional.layer_norm(x, (x.shape[1],), gn, ben, eps)
    return x, xn


def _tail_oracle_check(precision, ctx, Wp, bp, resid, W1, b1, W2, b2, g2, be2, gn, ben, x, xn=None, Wq=None, bq=None, qkv=None):
    """every element against the rounding-faithful float64 reference (tests/block_half_oracle.py) of the plain form"""
    nxt = "qkv" if Wq is not None else ("xn" if xn is not None else None)
    ops = BO.Operands(precision, ctx, Wp, bp, resid, W1, b1, W2, b2, g2, be2, gn, ben, Wq, bq, 1e-6, nxt=nxt)
    got = {k: v for k, v in (("x", x), ("xn", xn), ("qkv", qkv)) if v is not None}
    rep = BO.check_launch(ops, got)
    assert rep.ok(), str(rep)


@pytest.mark.parametrize("M,D,Hd", [(785, 384, 1536), (256, 384, 1536), (130, 128, 512), (1, 128, 128), (5000, 384, 1536), (80000, 384, 1536),
                                    (257, 128, 256), (40000, 128, 384), (60000, 128, 128)])   # odd chunk counts: the epilogue groups swap per item
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("with_next_ln", [True, False])
def test_block_tail(M, D, Hd, precision, with_next_ln):
    """proj + residual + norm2 + fc1 + GELU + fc2 + residual + next LayerNorm in one kernel: ragged row tiles, one and many items
    per CTA pair, both instantiated widths, with and without the trailing LayerNorm."""
    if not with_next_ln and M > 5000:
        pytest.skip("covered by the with_next_ln case")
    lib = vob._lib.load_library()
    eng = make_engine(precision=2 if precision == "fp16" else 0)
    dt = torch.float16 if precision == "fp16" else torch.bfloat16
    ctx = _rand((M, D), 80).to(dt)
    Wp = _rand((D, D), 81, 0.05).to(dt)
    W1 = _rand((Hd, D), 82, 0.06).to(dt)
    W2 = _rand((D, Hd), 83, 0.03).to(dt)
    bp, b1, b2 = _rand((D,), 84, 0.1), _rand((Hd,), 85, 0.2), _rand((D,), 86, 0.1)
    g2, be2 = _rand((D,), 87) * 0.1 + 1, _rand((D,), 88) * 0.1
    gn, ben = _rand((D,), 89) * 0.1 + 1, _rand((D,), 90) * 0.1
    resid = _rand((M, D), 91) * 2 + 0.5
    x = resid.clone()
    # the workspace's XN [M][2D]: only the first D columns are written
    xn = torch.full((M, 2 * D), float("nan"), device="cuda", dtype=dt)
    check(lib.vitocm_block_tail(eng, ptr(ctx), ctx.stride(0), ptr(Wp), Wp.stride(0), ptr(bp), ptr(g2), ptr(be2), ptr(W1), W1.stride(0), ptr(W2),
                                W2.stride(0), M, D, Hd, ptr(b1), ptr(b2), ptr(x), ptr(gn) if with_next_ln else None,
                                ptr(ben) if with_next_ln else None, ptr(xn), xn.stride(0), None, 0, None, None, 0, None, cur_stream()))
    torch.cuda.synchronize()
    ref_x, ref_xn = _tail_reference(ctx, Wp, bp, g2, be2, W1, b1, W2, b2, gn, ben, resid, dt)
    tol = 3e-3 if precision == "fp16" else 1.5e-2
    scale = (ref_x - resid).abs().max().item()
    err = (x - ref_x).abs().max().item()
    assert err <= tol * scale + 1e-4, (err, scale)
    if with_next_ln:
        assert torch.isnan(xn[:, D:].float()).all()
        got = xn[:, :D].float()
        assert torch.isfinite(got).all()
        # 16-bit rounding of the output + the error of x divided by the row's standard deviation
        tol_n = (2e-3 if precision == "fp16" else 1.2e-2) * ref_xn.abs().max().item() + 2 * tol * scale / ref_x.std(dim=1).min().item()
        assert (got - ref_xn).abs().max().item() <= tol_n
    else:
        assert torch.isnan(xn.float()).all()
    _tail_oracle_check(precision, ctx, Wp, bp, resid, W1, b1, W2, b2, g2, be2, gn, ben, x, xn[:, :D] if with_next_ln else None)


@pytest.mark.parametrize("M,D,Hd", [(785, 384, 1536), (130, 128, 512), (1, 128, 128), (5000, 384, 1536), (80000, 384, 1536), (257, 128, 256),
                                    (60000, 128, 128)])
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_block_tail_with_next_qkv(M, D, Hd, precision):
    """The block tail that also computes the NEXT block's QKV projection (the normalised rows never leave shared memory): X as before,
    QKV against the fp32 statement on the 16-bit rounded normalised rows; XN must stay untouched."""
    lib = vob._lib.load_library()
    eng = make_engine(precision=2 if precision == "fp16" else 0)
    dt = torch.float16 if precision == "fp16" else torch.bfloat16
    ctx = _rand((M, D), 120).to(dt)
    Wp = _rand((D, D), 121, 0.05).to(dt)
    W1 = _rand((Hd, D), 122, 0.06).to(dt)
    W2 = _rand((D, Hd), 123, 0.03).to(dt)
    Wq = _rand((3 * D, D), 124, 0.05).to(dt)
    bp, b1, b2, bq = _rand((D,), 125, 0.1), _rand((Hd,), 126, 0.2), _rand((D,), 127, 0.1), _rand((3 * D,), 128, 0.1)
    g2, be2 = _rand((D,), 129) * 0.1 + 1, _rand((D,), 130) * 0.1
    gn, ben = _rand((D,), 131) * 0.1 + 1, _rand((D,), 132) * 0.1
    resid = _rand((M, D), 133) * 2 + 0.5
    x = resid.clone()
    xn = torch.full((M, 2 * D), float("nan"), device="cuda", dtype=dt)
    qkv = torch.full((M, 3 * D), float("nan"), device="cuda", dtype=dt)
    check(lib.vitocm_block_tail(eng, ptr(ctx), ctx.stride(0), ptr(Wp), Wp.stride(0), ptr(bp), ptr(g2), ptr(be2), ptr(W1), W1.stride(0), ptr(W2),
                                W2.stride(0), M, D, Hd, ptr(b1), ptr(b2), ptr(x), ptr(gn), ptr(ben), ptr(xn), xn.stride(0), ptr(Wq), Wq.stride(0),
                                ptr(bq), ptr(qkv), qkv.stride(0), None, cur_stream()))
    torch.cuda.synchronize()
    ref_x, ref_xn = _tail_reference(ctx, Wp, bp, g2, be2, W1, b1, W2, b2, gn, ben, resid, dt)
    tol = 3e-3 if precision == "fp16" else 1.5e-2
    scale = (ref_x - resid).abs().max().item()
    assert (x - ref_x).abs().max().item() <= tol * scale + 1e-4
    assert torch.isnan(xn.float()).all()
    got = qkv.float()
    assert torch.isfinite(got).all()
    # from the kernel's own X (so that the error of X does not count twice): LayerNorm -> 16 bits -> Linear -> 16 bits
    xn_k = torch.nn.functional.layer_norm(x, (D,), gn, ben, 1e-6).to(dt).float()
    ref_q = xn_k @ Wq.float().T + bq
    err = (got - ref_q).abs().max().item()
    # one 16-bit ulp of the output + normalised rows that landed on the neighbouring 16-bit value (each worth |w| 2^-8 / 2^-11)
    assert err <= (6e-3 if precision == "fp16" else 4e-2) * ref_q.abs().max().item(), (err, ref_q.abs().max().item())
    assert (got - ref_q).abs().mean().item() <= (4e-4 if precision == "fp16" else 3e-3) * ref_q.abs().max().item()
    _tail_oracle_check(precision, ctx, Wp, bp, resid, W1, b1, W2, b2, g2, be2, gn, ben, x, Wq=Wq, bq=bq, qkv=qkv)


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_block_tail_statistics_with_large_means(precision):
    """LayerNorm statistics of the block tail (exact (mean, M2) per 32 values, Chan's combination across steps and warps) on rows
    whose mean is far from zero: offsets of 0 / 8 / 40 / 300 standard deviations, groups of 32 nearly equal large values and an
    exactly constant group -- the trailing LayerNorm must match torch's on the kernel's own X.  (Guards any cheaper form of the
    statistics: a one-sweep sum y^2 - n mean^2 without a fall-back fails here.)"""
    lib = vob._lib.load_library()
    eng = make_engine(precision=2 if precision == "fp16" else 0)
    dt = torch.float16 if precision == "fp16" else torch.bfloat16
    M, D, Hd = 1100, 384, 1536
    ctx = _rand((M, D), 140).to(dt)
    Wp = _rand((D, D), 141, 0.02).to(dt)
    W1 = _rand((Hd, D), 142, 0.06).to(dt)
    W2 = _rand((D, Hd), 143, 0.01).to(dt)
    bp, b1, b2 = _rand((D,), 144, 0.1), _rand((Hd,), 145, 0.2), _rand((D,), 146, 0.1)
    g2, be2 = _rand((D,), 147) * 0.1 + 1, _rand((D,), 148) * 0.1
    gn, ben = _rand((D,), 149) * 0.1 + 1, _rand((D,), 150) * 0.1
    resid = _rand((M, D), 151) * 0.5
    offs = torch.tensor([0.0, 4.0, 20.0, 150.0, -150.0], device="cuda")
    resid += offs[torch.arange(M, device="cuda") % 5][:, None]
    resid[7::11, 32:64] = 500.0 + 0.01 * _rand((len(range(7, M, 11)), 32), 152)    # one group far from the row's other values
    resid[3::13, 96:128] = -250.0                                                   # ... and an exactly constant one
    x = resid.clone()
    xn = torch.full((M, 2 * D), float("nan"), device="cuda", dtype=dt)
    check(lib.vitocm_block_tail(eng, ptr(ctx), ctx.stride(0), ptr(Wp), Wp.stride(0), ptr(bp), ptr(g2), ptr(be2), ptr(W1), W1.stride(0), ptr(W2),
                                W2.stride(0), M, D, Hd, ptr(b1), ptr(b2), ptr(x), ptr(gn), ptr(ben), ptr(xn), xn.stride(0), None, 0, None, None, 0,
                                None, cur_stream()))
    torch.cuda.synchronize()
    ref_x, _ = _tail_reference(ctx, Wp, bp, g2, be2, W1, b1, W2, b2, gn, ben, resid, dt)
    # X: norm2's statistics feed the MLP, so an error there shows as an error of the MLP's contribution
    scale = (ref_x - resid).abs().max().item()
    assert (x - ref_x).abs().max().item() <= (3e-3 if precision == "fp16" else 1.5e-2) * scale + 2e-4 * resid.abs().max().item()
    got = xn[:, :D].float()
    assert torch.isfinite(got).all()
    ref_n = torch.nn.functional.layer_norm(x.double(), (D,), gn.double(), ben.double(), 1e-6).float()
    err = (got - ref_n).abs()
    assert err.max().item() <= (2e-3 if precision == "fp16" else 1.2e-2) * ref_n.abs().max().item(), err.max().item()
    # per kind of row, so that a loss of accuracy confined to the offset rows cannot hide behind the others
    for k in range(5):
        rows = slice(k, M, 5)
        assert (err[rows].max() <= (2e-3 if precision == "fp16" else 1.2e-2) * ref_n[rows].abs().max()).item(), k
    _tail_oracle_check(precision, ctx, Wp, bp, resid, W1, b1, W2, b2, g2, be2, gn, ben, x, xn[:, :D])


def test_block_tail_matches_separate_kernels(engine):
    """The one-kernel block tail against the kernels it replaces (proj + LayerNorm GEMM, fused MLP, LayerNorm) on the same operands."""
    lib = vob._lib.load_library()
    M, D, Hd = 3000, 384, 1536
    dt = torch.bfloat16
    ctx = _rand((M, D), 100).to(dt)
    Wp = _rand((D, D), 101, 0.05).to(dt)
    W1 = _rand((Hd, D), 102, 0.06).to(dt)
    W2 = _rand((D, Hd), 103, 0.03).to(dt)
    bp, b1, b2 = _rand((D,), 104, 0.1), _rand((Hd,), 105, 0.2), _rand((D,), 106, 0.1)
    g2, be2 = _rand((D,), 107) * 0.1 + 1, _rand((D,), 108) * 0.1
    gn, ben = _rand((D,), 109) * 0.1 + 1, _rand((D,), 110) * 0.1
    resid = _rand((M, D), 111)
    x = resid.clone()
    xn = torch.zeros((M, 2 * D), device="cuda", dtype=dt)
    check(lib.vitocm_block_tail(engine, ptr(ctx), ctx.stride(0), ptr(Wp), Wp.stride(0), ptr(bp), ptr(g2), ptr(be2), ptr(W1), W1.stride(0), ptr(W2),
                                W2.stride(0), M, D, Hd, ptr(b1), ptr(b2), ptr(x), ptr(gn), ptr(ben), ptr(xn), xn.stride(0), None, 0, None, None, 0, None, cur_stream()))
    y = resid.clone()
    yn = torch.zeros((M, 2 * D), device="cuda", dtype=dt)
    check(lib.vitocm_gemm_ln(engine, ptr(ctx), ctx.stride(0), ptr(Wp), Wp.stride(0), M, D, D, ptr(bp), ptr(y), ptr(g2), ptr(be2), ptr(yn),
                             yn.stride(0), cur_stream()))
    check(lib.vitocm_mlp_fused(engine, ptr(yn), yn.stride(0), ptr(W1), W1.stride(0), ptr(W2), W2.stride(0), M, D, Hd, ptr(b1), ptr(b2), ptr(y),
                               cur_stream()))
    torch.cuda.synchronize()
    scale = (y - resid).abs().max().item()
    # norm2's rows are rounded to bf16 in both paths, from statistics summed in a different order: a few of them land on the
    # neighbouring bf16 value
    assert (x - y).abs().max().item() <= 4e-3 * scale
    assert (x - y).abs().mean().item() <= 1e-4 * scale
    ref_n = torch.nn.functional.layer_norm(y, (D,), gn, ben, 1e-6)
    assert (xn[:, :D].float() - ref_n).abs().max().item() <= 1.5e-2 * ref_n.abs().max().item()


def test_mlp_fused_matches_separate_gemms(engine):
    """The fused kernel against the two-GEMM path it replaces (same operands, same GELU form): only the summation order differs."""
    lib = vob._lib.load_library()
    M, D, Hd = 3000, 384, 1536
    A = _rand((M, D), 70).to(torch.bfloat16)
    W1 = _rand((Hd, D), 71, 0.06).to(torch.bfloat16)
    W2 = _rand((D, Hd), 72, 0.03).to(torch.bfloat16)
    b1, b2 = _rand((Hd,), 73, 0.2), _rand((D,), 74, 0.1)
    resid = _rand((M, D), 75)
    x = resid.clone()
    check(lib.vitocm_mlp_fused(engine, ptr(A), A.stride(0), ptr(W1), W1.stride(0), ptr(W2), W2.stride(0), M, D, Hd, ptr(b1), ptr(b2), ptr(x),
                               cur_stream()))
    hid = torch.empty(M, Hd, device="cuda", dtype=torch.bfloat16)
    gemm(engine, A, W1, M, Hd, D, 0, 1, b1, hid, Hd)
    y = resid.clone()
    gemm(engine, hid, W2, M, D, Hd, 0, 2, b2, y, D)
    torch.cuda.synchronize()
    assert (x - y).abs().max().item() <= 2e-4 * (y - resid).abs().max().item() + 1e-5
