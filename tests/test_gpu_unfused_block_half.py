"""GPU (B200): the unfused second half of a block -- the path the forward takes where the block tail has no instantiation (ViT-B,
D = 768) -- stage by stage, element by element, against the float64 stage references of tests/block_half_oracle.py:

    layernorm_kernel (norm1)  ->  QKV GEMM (bias, 16 bits, CTA pairs, BN 256)
    proj GEMM (bias, TMA reduce-add into a pre-filled X)  ->  layernorm_kernel (norm2)
    fc1 GEMM (bias, GELU, 16 bits, CTA pairs, BN 192)  ->  fc2 GEMM (bias, reduce-add into X, CTA pairs, BN 256)

Each stage reads the exact output of the kernel before it (so its reference reads the same 16-bit and fp32 values) and is checked on
every row: a 16-bit output must lie in [RN16(v - w), RN16(v + w)], an fp32 output within w of v.  Launches of 137 375 rows (175 tiles
of 785) and 1 607 680 rows (a full chunk of 2 048 tiles: 4.9 GB of fp32 X, 7.4 GB of QKV), bf16 and fp16 engines.  Outputs carry NaN
guard rows after M and NaN guard columns beyond N of their pitch; the A operands are read through wider pitches whose extra columns hold
NaN.  At D = 384 the same stages run at 137 375 rows, and the block tail runs on the same operands against the block-half reference:
the two references agree on the one value both compute from the same inputs (the proj + residual rows y)."""
import time

import pytest
import torch

import block_half_oracle as BO
import vitocm_b200 as vob
from gpu_util import make_engine
from vitocm_b200._lib import check, cur_stream, ptr

pytestmark = pytest.mark.gpu

G = 64          # guard rows / columns
CHUNK = 16384   # rows per float64 reference chunk


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


def _nan(rows, cols, dt):
    return torch.full((rows, cols), float("nan"), device="cuda", dtype=dt)


def _rand(shape, g, scale=1.0):
    return torch.randn(shape, generator=g, device="cuda") * scale


def _gemm(eng, A, lda, W, M, N, K, epi, bias, out, ldo):
    lib = vob._lib.load_library()
    check(lib.vitocm_gemm(eng, ptr(A), lda, ptr(W), W.stride(0), M, N, K, 0, epi, ptr(bias), ptr(out), ldo, 0, 0, cur_stream()))
    torch.cuda.synchronize()


def _layernorm(eng, X, g, b, out, ldo, M):
    lib = vob._lib.load_library()
    check(lib.vitocm_layernorm(eng, ptr(X), ptr(g), ptr(b), ptr(out), ldo, 0, 0, M, cur_stream()))
    torch.cuda.synchronize()


def _check(rep, name, M, got, ref_fn, prec):
    """every row of got [M][N] against ref_fn(row slice) -> (v, w), chunked"""
    for s in range(0, M, CHUNK):
        e = min(M, s + CHUNK)
        v, w = ref_fn(slice(s, e))
        rep.add(name, torch.arange(s, e, device="cuda"), got[s:e], v, w, prec)


def _nan_guards(t, rows, cols, what):
    assert torch.isnan(t[rows:].float()).all(), f"{what}: a guard row was written"
    assert torch.isnan(t[:rows, cols:].float()).all(), f"{what}: a guard column was written"


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("D,M", [(768, 137375), (768, 1607680), (384, 137375)])
def test_unfused_block_half_stages(prec, D, M):
    t0 = time.time()
    dt = BO.DT[prec]
    Hd = 4 * D
    eng = make_engine(embed_dim=D, heads=D // 64, hidden=Hd, precision=2 if prec == "fp16" else 0)
    lib = vob._lib.load_library()
    g = torch.Generator(device="cuda").manual_seed(700 + D + M % 1000)
    q16 = lambda t: BO.rn16(t, prec)
    g1, be1, g2, be2 = 1 + _rand(D, g, 0.1), _rand(D, g, 0.1), 1 + _rand(D, g, 0.1), _rand(D, g, 0.1)
    Wq, bq = q16(_rand((3 * D, D), g, D ** -0.5)), _rand(3 * D, g, 0.1)
    Wp, bp = q16(_rand((D, D), g, 0.5 * D ** -0.5)), _rand(D, g, 0.1)
    W1, b1 = q16(_rand((Hd, D), g, 3.0 * D ** -0.5)), _rand(Hd, g, 0.2)     # pre-activations of std ~3: both GELU tails
    W2, b2 = q16(_rand((D, Hd), g, Hd ** -0.5)), _rand(D, g, 0.1)
    rep = BO.Report()
    try:
        # -------- norm1: rows offset by 0 / 20 / -150 standard deviations
        X0 = _rand((M, D), g, 1.5) + 0.5
        X0 += torch.tensor([0.0, 20.0, 0.0, -150.0, 0.0], device="cuda")[torch.arange(M, device="cuda") % 5][:, None]
        XN = _nan(M + G, 2 * D, dt)                        # the workspace's XN [M][2D]: columns D.. are not written
        _layernorm(eng, X0, g1, be1, XN, 2 * D, M)
        _nan_guards(XN, M, D, "norm1")
        _check(rep, "norm1", M, XN[:M, :D], lambda r: BO.stage_layernorm(X0[r], g1, be1), prec)
        # -------- QKV GEMM on the kernel's own XN (read through its 2D pitch)
        QKV = _nan(M + G, 3 * D + G, dt)
        _gemm(eng, XN, 2 * D, Wq, M, 3 * D, D, 0, bq, QKV, 3 * D + G)
        _nan_guards(QKV, M, 3 * D, "qkv")
        _check(rep, "qkv", M, QKV[:M, :3 * D], lambda r: BO.stage_linear(XN[r, :D], Wq, bq), prec)
        del QKV, XN
        # -------- proj: X += CTX . Wp^T + bp (reduce-add into a pre-filled X with guard rows / columns)
        CTX = _nan(M, D + G, dt)
        CTX[:, :D] = q16(_rand((M, D), g))
        X = _nan(M + G, D + 32, torch.float32)
        X[:M, :D] = X0
        _gemm(eng, CTX, D + G, Wp, M, D, D, 2, bp, X, D + 32)
        _nan_guards(X, M, D, "proj")
        _check(rep, "proj", M, X[:M, :D], lambda r: BO.stage_reduce_add(X0[r], CTX[r, :D], Wp, bp), None)
        if D == 384:   # cross-check: the block-half reference computes the same float64 rows y from the same inputs
            ref = BO.Operands(prec, CTX[:, :D], Wp, bp, X0, W1, b1, W2, b2, g2, be2, eps=1e-6)
            rows = torch.arange(0, M, 997, device="cuda")
            y_tail = ref.rows(rows)["y"][0]
            y_stage = BO.stage_reduce_add(X0[rows], CTX[rows, :D], Wp, bp)[0]
            assert torch.allclose(y_tail, y_stage, rtol=0, atol=1e-12 * (1 + y_stage.abs().max().item()))
            Xt = X0.clone()   # ... and the block tail on the same operands, against it
            check(lib.vitocm_block_tail(eng, ptr(CTX), CTX.stride(0), ptr(Wp), D, ptr(bp), ptr(g2), ptr(be2), ptr(W1), D, ptr(W2), Hd, M, D,
                                        Hd, ptr(b1), ptr(b2), ptr(Xt), None, None, None, 0, None, 0, None, None, 0, None, cur_stream()))
            torch.cuda.synchronize()
            rep_tail = BO.check_launch(ref, {"x": Xt})
            assert rep_tail.ok(), f"block tail on the unfused test's operands: {rep_tail}"
            del Xt
        Y = X[:M, :D].contiguous()
        del X
        # -------- norm2 on the kernel's own residual rows
        XN2 = _nan(M + G, 2 * D, dt)
        _layernorm(eng, Y, g2, be2, XN2, 2 * D, M)
        _nan_guards(XN2, M, D, "norm2")
        _check(rep, "norm2", M, XN2[:M, :D], lambda r: BO.stage_layernorm(Y[r], g2, be2), prec)
        # -------- fc1 + GELU
        H = _nan(M + G, Hd + G, dt)
        _gemm(eng, XN2, 2 * D, W1, M, Hd, D, 1, b1, H, Hd + G)
        _nan_guards(H, M, Hd, "fc1")
        _check(rep, "fc1", M, H[:M, :Hd], lambda r: BO.stage_gelu(XN2[r, :D], W1, b1, prec), prec)
        del XN2
        # -------- fc2: X += H . W2^T + b2 on the residual rows proj left (H read through its wider pitch)
        X2 = _nan(M + G, D + 32, torch.float32)
        X2[:M, :D] = Y
        _gemm(eng, H, Hd + G, W2, M, D, Hd, 2, b2, X2, D + 32)
        _nan_guards(X2, M, D, "fc2")
        _check(rep, "fc2", M, X2[:M, :D], lambda r: BO.stage_reduce_add(Y[r], H[r, :Hd], W2, b2), None)
        del H, X2
        assert rep.ok(), str(rep)
        print(f"\nunfused {prec} D={D} M={M}: every row checked; {rep}  [{time.time() - t0:.1f} s]")
    finally:
        lib.vitocm_destroy(eng)
