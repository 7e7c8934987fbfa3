"""GPU (B200): the training step's kernels one by one -- the fc1 epilogue that also saves the GELU input, the input-gradient epilogue
through the GELU (both on every tile path, CTA pairs included), the LayerNorm backward and the MIM loss backward -- each against a
float64 statement of the same operation on the same 16-bit operands, plus the clip and AdamW kernels.

Bounds are per element and follow from the arithmetic: half an ulp of the 16-bit output, fp32 accumulation (about
K 2^-24 sum |a| |b|), and the documented error of each GELU form (gemm_sm100.cuh).  Outputs are pre-filled with NaN and carry pad
rows and pad columns that must stay NaN, so that an error confined to one tile, or a store one tile off, fails."""
import math

import numpy as np
import pytest
import torch

import vitocm_b200 as vob
from gpu_util import gemm, make_engine
from vitocm_b200._lib import check, cur_stream, ptr

pytestmark = pytest.mark.gpu

FP16 = 2
EPS24 = 2.0 ** -24
# documented maximum errors of the sigmoid-form GELU and of its derivative (gemm_sm100.cuh): bf16 engines use the three-coefficient
# form, fp16 engines the five-coefficient one
GELU_ERR = {"bf16": 2.5e-5, "fp16": 3.0e-6}
DGELU_ERR = {"bf16": 1.1e-4, "fp16": 1.5e-5}
DT = {"bf16": torch.bfloat16, "fp16": torch.float16}
MANT = {"bf16": 7, "fp16": 10}        # stored significand bits
EMIN = {"bf16": -126, "fp16": -14}    # exponent of the smallest normal value
PAD = 64


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


def ulp16(x, prec):
    """ulp of the 16-bit format at |x| (float64 tensor), subnormal spacing below the smallest normal"""
    _, ex = torch.frexp(x.abs())
    e = torch.where(x == 0, EMIN[prec], torch.clamp(ex.to(torch.float64) - 1, min=EMIN[prec]))
    return torch.pow(2.0, e - MANT[prec])


def gelu64(x):
    return 0.5 * x * (1.0 + torch.special.erf(x / math.sqrt(2.0)))


def dgelu64(x):
    """d/dx of x Phi(x), erf form: Phi(x) + x phi(x)"""
    return 0.5 * (1.0 + torch.special.erf(x / math.sqrt(2.0))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2.0 * math.pi)


def _assert_within(got, ref, bound, what):
    err = (got - ref).abs()
    bad = ~(err <= bound)                 # NaN fails too
    if bad.any():
        idx = bad.nonzero()[0].tolist()
        pytest.fail(f"{what}: {int(bad.sum())} elements out of bound, first at {idx}: got {got[tuple(idx)].item():.9g} "
                    f"ref {ref[tuple(idx)].item():.9g} bound {bound[tuple(idx)].item():.3g}")
    return (err / bound).max().item()


def _assert_nan(t, what):
    assert torch.isnan(t.float()).all(), f"{what}: a pad element was written"


# ------------------------------------------------------------------------------------------------------------ tile paths
def _pick_bn(M, N, sms, max_bn=256):
    """pick_bn of vitocm_api.cu"""
    tiles_m = (M + 127) // 128
    best, best_cost = 0, 0
    for bn in (256, 192, 128, 64):
        if bn > max_bn or N % bn:
            continue
        cost = ((tiles_m * (N // bn) + sms - 1) // sms) * (bn + 48)
        if best == 0 or cost < best_cost:
            best, best_cost = bn, cost
    return best


def gelu_epilogue_path(M, N, K, sms):
    """The GEMM run_gemm launches for the two GELU epilogues (single 16-bit operands; no resident weight panel for either)."""
    if (M >= 65536 or (K >= 1024 and M >= 4096)) and M >= 512 and (N % 256 == 0 or N % 192 == 0 or N % 128 == 0):
        bn = 192 if N % 192 == 0 else (256 if N % 256 == 0 else 128)
        return f"pair-bn{bn}"
    return f"bn{_pick_bn(M, N, sms)}"


# (M, N = hidden, K = embed_dim): every tile width, 12 epilogue warps (BN 192), many tiles per CTA, CTA pairs at each width, and
# ragged pair tiles (one live row in the last pair; 129 rows in it)
PATHS = [(128, 1536, 384, "bn64"), (785, 1536, 384, "bn128"), (1570, 1536, 384, "bn192"), (25120, 1536, 384, "bn256"),
         (70000, 1536, 384, "pair-bn192"), (66000, 512, 128, "pair-bn256"), (70000, 640, 384, "pair-bn128"),
         (65537, 3072, 768, "pair-bn192"), (65537, 1536, 384, "pair-bn192"), (65536 + 129, 1536, 384, "pair-bn192")]
PATH_PARAMS = [pytest.param(M, N, K, path, id=f"{path}-M{M}-N{N}-K{K}") for M, N, K, path in PATHS]


def _check_path(M, N, K, path):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if sms == 148:   # the B200: the test id names the path the selection rule takes
        assert gelu_epilogue_path(M, N, K, sms) == path


def _fc1_operands(M, N, K, prec, seed):
    dt = DT[prec]
    A = _rand((M, K), seed).to(dt)
    W = _rand((N, K), seed + 1, 3.0 / math.sqrt(K)).to(dt)     # pre-activations of std ~3: both GELU tails are populated
    b = _rand((N,), seed + 2, 0.5)
    return A, W, b


def _fc1_reference(A, W, b):
    pre = A.double() @ W.double().T + b.double()
    mag = A.double().abs() @ W.double().abs().T + b.double().abs()
    return pre, (A.shape[1] + 2) * EPS24 * mag          # fp32 accumulation


def _run_fc1(eng, A, W, b, HP, ldo, M, N, K):
    gemm(eng, A, W, M, N, K, 0, 1, b, HP, ldo, 2, N)


def _check_fc1(HP, pre_ref, acc_err, prec, N, what):
    pre_k = HP[:, N:2 * N].double()
    r_pre = _assert_within(pre_k, pre_ref, 0.5 * ulp16(torch.maximum(pre_k.abs(), pre_ref.abs()), prec) + acc_err, f"{what} pre")
    g_k = HP[:, :N].double()
    g_ref = gelu64(pre_ref)
    bound = 0.5 * ulp16(torch.maximum(g_k.abs(), g_ref.abs()), prec) + GELU_ERR[prec] + 2.0 ** -21 * pre_ref.abs() + 1.13 * acc_err
    r_gelu = _assert_within(g_k, g_ref, bound, f"{what} gelu")
    return r_pre, r_gelu


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("M,N,K,path", PATH_PARAMS)
def test_fc1_saves_pre_activation(engines, prec, M, N, K, path):
    """Epilogue 1 with split_out 2 (the training fc1): out[:, :N] = gelu(pre), out[:, N:2N] = pre = 16-bit(acc + bias)."""
    _check_path(M, N, K, path)
    A, W, b = _fc1_operands(M, N, K, prec, 100 + M % 97)
    ldo = 2 * N + PAD
    HP = torch.full((M + PAD, ldo), float("nan"), device="cuda", dtype=DT[prec])
    _run_fc1(engines[prec], A, W, b, HP, ldo, M, N, K)
    pre_ref, acc_err = _fc1_reference(A, W, b)
    r = _check_fc1(HP[:M], pre_ref, acc_err, prec, N, path)
    _assert_nan(HP[:M, 2 * N:], "pad columns")
    _assert_nan(HP[M:], "pad rows")
    print(f"\nfc1 {prec} {path} M={M}: worst error / bound  pre {r[0]:.3f}  gelu {r[1]:.3f}")


def _dgelu(eng, dY, Wt, M, N, K, pre, ld_pre, out, ldo):
    lib = vob._lib.load_library()
    check(lib.vitocm_gemm_dgelu(eng, ptr(dY), dY.stride(0), ptr(Wt), Wt.stride(0), M, N, K, pre.data_ptr(), ld_pre, ptr(out), ldo,
                                cur_stream()))
    torch.cuda.synchronize()


def _dgelu_bound(out_k, ref, acc, acc_err, prec):
    """16-bit rounding of the output, the derivative form's error times |acc|, gelu' (<= 1.13) times the accumulation error"""
    return (0.5 * ulp16(torch.maximum(out_k.abs(), ref.abs()), prec) + acc.abs() * (DGELU_ERR[prec] + 1e-6) + 1.13 * acc_err)


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
def test_dgelu_every_16bit_input(engines, prec):
    """The accumulator is exactly 1 (one-hot A, B's first column all ones), so out = 16-bit(gelu'(pre)) for every finite 16-bit pre:
    +-0, subnormals, the tails beyond |x| = 10 where the bf16 form clamps u, +-65504 and the largest bf16 values.  Every output is
    finite and within half an ulp plus the documented error of the derivative form of the exact erf derivative."""
    dt = DT[prec]
    bits = torch.arange(65536, device="cuda", dtype=torch.int32).to(torch.int16).view(dt)
    vals = bits[torch.isfinite(bits.float())]
    M, N, K = 256, 256, 64
    pre = torch.zeros(M * N, device="cuda", dtype=dt)
    pre[:vals.numel()] = vals
    pre = pre.reshape(M, N)
    A = torch.zeros(M, K, device="cuda", dtype=dt)
    A[:, 0] = 1
    B = torch.zeros(N, K, device="cuda", dtype=dt)
    B[:, 0] = 1
    out = torch.full((M + PAD, N + PAD), float("nan"), device="cuda", dtype=dt)
    _dgelu(engines[prec], A, B, M, N, K, pre, N, out, N + PAD)
    got = out[:M, :N].double()
    assert torch.isfinite(got).all(), pre.flatten()[~torch.isfinite(got.flatten())][:8].tolist()
    ref = dgelu64(pre.double())
    one = torch.ones_like(ref)
    r = _assert_within(got, ref, _dgelu_bound(got, ref, one, 0 * one, prec), "gelu'")
    assert vals.numel() == 65536 - 2 ** (MANT[prec] + 1)              # every pattern but +-inf and the NaNs
    assert pre.float().max().item() == torch.finfo(dt).max and pre.float().min().item() == -torch.finfo(dt).max
    _assert_nan(out[:M, N:], "pad columns")
    _assert_nan(out[M:], "pad rows")
    print(f"\ndgelu sweep {prec}: {vals.numel()} finite inputs, worst error / bound {r:.3f}")


def _dgelu_operands(M, N, K, prec, seed):
    dt = DT[prec]
    dY = _rand((M, K), seed, 0.5).to(dt)
    Wt = _rand((N, K), seed + 1, 1.0 / math.sqrt(K)).to(dt)
    return dY, Wt


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("M,N,K,path", PATH_PARAMS)
def test_dgelu_random_operands(engines, prec, M, N, K, path):
    """dPRE = (dY . Wt^T) * gelu'(pre), pre read at HP + N with ld_pre = 2N as in the step; HP[:, :N] holds NaN, so a wrong column
    offset of the pre-activation box shows as NaN, a wrong row (CTA pairs) as a wrong value."""
    _check_path(M, N, K, path)
    dt = DT[prec]
    dY, Wt = _dgelu_operands(M, N, K, prec, 200 + M % 89)
    HP = torch.full((M, 2 * N), float("nan"), device="cuda", dtype=dt)
    HP[:, N:] = _rand((M, N), 203, 3.0).to(dt)
    out = torch.full((M + PAD, N + PAD), float("nan"), device="cuda", dtype=dt)
    _dgelu(engines[prec], dY, Wt, M, N, K, HP[:, N:], 2 * N, out, N + PAD)
    acc = dY.double() @ Wt.double().T
    acc_err = (K + 2) * EPS24 * (dY.double().abs() @ Wt.double().abs().T)
    pre = HP[:, N:].double()
    ref = acc * dgelu64(pre)
    got = out[:M, :N].double()
    r = _assert_within(got, ref, _dgelu_bound(got, ref, acc, acc_err, prec), f"dgelu {path}")
    _assert_nan(out[:M, N:], "pad columns")
    _assert_nan(out[M:], "pad rows")
    print(f"\ndgelu {prec} {path} M={M}: worst error / bound {r:.3f}")


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("M,N,K", [(785, 1536, 384), (70000, 1536, 384), (66000, 512, 128)])
def test_fc1_then_dgelu_chain_matches_autograd(engines, prec, M, N, K):
    """The step's own buffer: fc1 writes HP = gelu | pre (ldo 2N), the input-gradient GEMM reads pre from HP + N.  Against float64
    autograd of gelu(XN W1^T + b1) for the upstream dH = dY Wt^T."""
    dt = DT[prec]
    A, W, b = _fc1_operands(M, N, K, prec, 300)
    dY, Wt = _dgelu_operands(M, N, K, prec, 310)
    HP = torch.full((M + PAD, 2 * N), float("nan"), device="cuda", dtype=dt)
    _run_fc1(engines[prec], A, W, b, HP, 2 * N, M, N, K)
    _assert_nan(HP[M:], "pad rows of HP")
    out = torch.full((M + PAD, N + PAD), float("nan"), device="cuda", dtype=dt)
    _dgelu(engines[prec], dY, Wt, M, N, K, HP[:M, N:], 2 * N, out, N + PAD)
    pre64 = (A.double() @ W.double().T + b.double()).requires_grad_(True)
    acc = dY.double() @ Wt.double().T
    gelu64(pre64).backward(acc)
    ref = pre64.grad
    pre_ref = pre64.detach()
    _, fc1_err = _fc1_reference(A, W, b)
    acc_err = (K + 2) * EPS24 * (dY.double().abs() @ Wt.double().abs().T)
    got = out[:M, :N].double()
    # the saved pre-activation is 16-bit: |gelu''| <= 0.8 times its rounding and accumulation error
    pre_err = ulp16(pre_ref, prec) + fc1_err
    bound = _dgelu_bound(got, ref, acc, acc_err, prec) + 0.8 * acc.abs() * pre_err
    r = _assert_within(got, ref, bound, "chain")
    _assert_nan(out[:M, N:], "pad columns")
    _assert_nan(out[M:], "pad rows")
    print(f"\nfc1 -> dgelu chain {prec} M={M} N={N}: worst error / bound {r:.3f}")


# ------------------------------------------------------------------------------------------------------------ LayerNorm backward
def _ln_bwd(eng, X, dy_buf, ld_dy, gamma, dX, dXb, dgamma, dbeta, dbias, accumulate, M, D, lscale):
    lib = vob._lib.load_library()
    check(lib.vitocm_layernorm_bwd(eng, ptr(X), ptr(dy_buf), ld_dy, ptr(gamma), ptr(dX), ptr(dXb), ptr(dgamma), ptr(dbeta), ptr(dbias),
                                   accumulate, M, D, ptr(lscale), cur_stream()))
    torch.cuda.synchronize()


def _ln_rows(M, D, seed):
    """rows of std 0.7 offset by 0, 4, 20, +-150 standard deviations; every 13th row exactly constant"""
    x = _rand((M, D), seed, 0.7)
    offs = torch.tensor([0.0, 4.0, 20.0, 150.0, -150.0], device="cuda") * 0.7
    x += offs[torch.arange(M, device="cuda") % 5][:, None]
    x[12::13] = -2.5
    return x


def _ln_reference(X, dy, gamma):
    """float64 autograd of layer_norm(X) for the upstream dy, and the row quantities the error bounds use"""
    D = X.shape[1]
    X64 = X.double().requires_grad_(True)
    g64 = gamma.double().requires_grad_(True)
    b64 = torch.zeros(D, dtype=torch.float64, device="cuda", requires_grad=True)
    torch.nn.functional.layer_norm(X64, (D,), g64, b64, 1e-6).backward(dy.double())
    with torch.no_grad():
        mean = X64.mean(1, keepdim=True)
        rstd = 1.0 / torch.sqrt(((X64 - mean) ** 2).mean(1, keepdim=True) + 1e-6)
        xhat = (X64 - mean) * rstd
    return X64.grad, g64.grad, b64.grad, mean, rstd, xhat


KC = 128   # fp32 row statistics and dot products over D <= 1024 (32 values per lane, then a 5-level shuffle tree), with room


def _ln_dx_bound(dy64, gamma, mean, rstd, xhat):
    """|dx_kernel - dx| per element: rstd (g - mean g - xhat mean(g xhat)) evaluated in fp32; the fp32 row mean's error is
    amplified by the row's normalised offset |mean| rstd (and the resulting xhat error enters through mean(g xhat))."""
    g = dy64 * gamma.double()
    mg = g.abs().mean(1, keepdim=True)
    mgx = (g * xhat).abs().mean(1, keepdim=True)
    amp = 1.0 + mean.abs() * rstd
    return KC * EPS24 * rstd * (g.abs() + mg + xhat.abs() * mgx + amp * (mgx + xhat.abs() * mg))


def _ln_case_check(prec, M, D, X, dy, gamma, ref, dX_in, accumulate, dX, dXb, sums0, sums, with_bias):
    dx_ref, dg_ref, db_ref, mean, rstd, xhat = ref
    dy64 = dy.double()
    grid = min((M + 63) // 64, 296)
    n_add = (M + grid * 8 - 1) // (grid * 8) + 8 + grid + 2       # fp32 additions along one column sum, worst case
    dX_ref = dx_ref + (dX_in.double() if accumulate else 0.0)
    bdx = _ln_dx_bound(dy64, gamma, mean, rstd, xhat) + EPS24 * dX_ref.abs()
    ratios = {"dX": _assert_within(dX.double(), dX_ref, bdx, f"dX acc={accumulate}")}
    # the 16-bit copy is the round-to-nearest conversion of the kernel's own dX (fp16: saturating at 65504)
    want = dX.clamp(-65504, 65504).half() if prec == "fp16" else dX.to(torch.bfloat16)
    assert torch.equal(dXb.view(torch.int16), want.view(torch.int16)), "dXb is not the 16-bit rounding of dX"
    dxh_err = KC * EPS24 * (xhat.abs() + 1.0 + mean.abs() * rstd)
    g0, b0, o0 = sums0
    dg, db, do = sums
    bg = n_add * EPS24 * (g0.double().abs() + (dy64 * xhat).abs().sum(0)) + (dy64.abs() * dxh_err).sum(0)
    ratios["dgamma"] = _assert_within(dg.double(), g0.double() + dg_ref, bg, "dgamma")
    bb = n_add * EPS24 * (b0.double().abs() + dy64.abs().sum(0))
    ratios["dbeta"] = _assert_within(db.double(), b0.double() + db_ref, bb, "dbeta")
    if with_bias:
        bo = n_add * EPS24 * (o0.double().abs() + dX_ref.abs().sum(0)) + bdx.sum(0)
        ratios["dbias"] = _assert_within(do.double(), o0.double() + dX_ref.sum(0), bo, "dbias_out (column sums of the new dX)")
    else:
        assert torch.equal(do, o0), "dbias_out was NULL: the buffer must not change"
    return ratios


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("D", [128, 384, 768, 192, 256, 1024])
@pytest.mark.parametrize("M", [1, 63, 64, 65, 785, 25120, 100000])
def test_layernorm_backward(engines, prec, D, M):
    """ln_bwd_kernel (NV = 1, 3, 6 and the generic NV = 0 for D = 192, 256, 1024) against float64 autograd of layer_norm:
    dX = (accumulate ? dX_in : 0) + dx, dXb = 16-bit(dX), dgamma / dbeta accumulated onto non-zero buffers, dbias_out += column
    sums of the NEW dX (NULL: untouched); dy at pitch D and 3D (the other columns NaN); rows far from zero and constant rows."""
    dt = DT[prec]
    eng = engines[prec]
    X = _ln_rows(M, D, 400 + D)
    gamma = _rand((D,), 401) * 0.1 + 1.0
    dy = _rand((M, D), 402, 0.5).to(dt)
    ref = _ln_reference(X, dy, gamma)
    lscale = torch.ones(2, device="cuda") if prec == "fp16" else None
    worst = {}
    for accumulate, with_bias, ld_dy in ((1, True, 3 * D), (0, True, D), (1, False, D)):
        dy_buf = torch.full((M, ld_dy), float("nan"), device="cuda", dtype=dt)
        dy_buf[:, :D] = dy
        dX_in = _rand((M, D), 403 + accumulate, 2.0)
        dX = dX_in.clone()
        dXb = torch.full((M + PAD, D), float("nan"), device="cuda", dtype=dt)
        sums0 = tuple(_rand((D,), 410 + k) for k in range(3))
        sums = tuple(s.clone() for s in sums0)
        _ln_bwd(eng, X, dy_buf, ld_dy, gamma, dX, dXb, sums[0], sums[1], sums[2] if with_bias else None, accumulate, M, D, lscale)
        _assert_nan(dXb[M:], "pad rows of dXb")
        r = _ln_case_check(prec, M, D, X, dy, gamma, ref, dX_in, accumulate, dX, dXb[:M], sums0, sums, with_bias)
        for k, v in r.items():
            worst[k] = max(worst.get(k, 0.0), v)
    print(f"\nln_bwd {prec} D={D} M={M}: worst error / bound " + "  ".join(f"{k} {v:.3f}" for k, v in worst.items()))


@pytest.mark.parametrize("D", [128, 384, 768, 192, 256, 1024])
@pytest.mark.parametrize("accumulate", [0, 1])
def test_layernorm_backward_fp16_loss_scale(engines, D, accumulate):
    """fp16 engines: dy and dX carry the loss scale S.  dX from S dy (and S dX_in) with lscale = [S, 1/S] is bit-equal to S times
    dX from dy with lscale = [1, 1]; dgamma, dbeta and dbias_out come out unscaled (atomics: within tolerance)."""
    M, S = 25120, 2.0 ** 10
    eng = engines["fp16"]
    X = _ln_rows(M, D, 500 + D)
    gamma = _rand((D,), 501) * 0.1 + 1.0
    dy = _rand((M, D), 502, 0.5).half()
    dX_in = _rand((M, D), 503, 2.0)
    out = {}
    for s in (1.0, S):
        dX = dX_in * s
        dXb = torch.empty(M, D, device="cuda", dtype=torch.float16)
        sums = tuple(torch.zeros(D, device="cuda") for _ in range(3))
        _ln_bwd(eng, X, (dy.float() * s).half(), D, gamma, dX, dXb, *sums, accumulate, M, D, torch.tensor([s, 1.0 / s], device="cuda"))
        out[s] = (dX, dXb, sums)
    assert torch.equal(out[S][0], out[1.0][0] * S), "scaled dX is not S x the unscaled dX"
    assert torch.equal(out[S][1].view(torch.int16), out[S][0].clamp(-65504, 65504).half().view(torch.int16))
    xhat = _ln_reference(X, dy, gamma)[5]
    grid = min((M + 63) // 64, 296)
    n_add = (M + grid * 8 - 1) // (grid * 8) + 8 + grid + 2
    dy64 = dy.double()
    # both runs sum the same per-lane partials (exactly scaled); only the order of the atomics may differ
    bounds = (2 * n_add * EPS24 * (dy64 * xhat).abs().sum(0), 2 * n_add * EPS24 * dy64.abs().sum(0),
              2 * n_add * EPS24 * out[1.0][0].double().abs().sum(0))
    for name, a, b, bound in zip(("dgamma", "dbeta", "dbias_out"), out[S][2], out[1.0][2], bounds):
        _assert_within(a.double(), b.double(), bound, f"{name} under the loss scale")


# ------------------------------------------------------------------------------------------------------------ MIM loss backward
def _loss_scale_rule(coef):
    """include/vitocm.h / loss_scale_exp: S = 2^e with |coef| S in [1, 2), e clamped to +-126; S = 1 for 0, inf and NaN"""
    c = float(coef)
    if c == 0.0 or not math.isfinite(c):
        return 0
    _, ex = math.frexp(abs(c))
    return max(-126, min(126, 1 - ex))


def _mim_inputs(B, C, H, W, p, seed, mask_p=0.6):
    rs = np.random.RandomState(seed)
    n = (H // p) * (W // p)
    mask = (rs.rand(B, n) < mask_p).astype(np.float32)
    Y = rs.randn(B, C * p * p, H // p, W // p).astype(np.float32)
    x_rec = np.ascontiguousarray(torch.nn.functional.pixel_shuffle(torch.from_numpy(Y), p).numpy())
    x = x_rec + rs.randn(*x_rec.shape).astype(np.float32)
    ties = rs.rand(*x.shape) < 0.15
    x[ties] = x_rec[ties]                                        # d = 0: the gradient of |d| is 0 there
    return x, x_rec, mask, Y


def _mim_kernel_numpy(x, x_rec, mask, sums1, gscale, C, p, f16):
    """the kernel's formula in float32: coef = gscale / (f32(sums[1] + 1e-5) C), times S on fp16; +-mask coef, 0 at ties, CLS rows 0"""
    B, _, H, W = x.shape
    Hp, Wp = H // p, W // p
    with np.errstate(over="ignore"):                                              # 2^112 / (1e-5 C) overflows to inf at C = 1
        coef = np.float32(gscale) / (np.float32(sums1 + 1e-5) * np.float32(C))
    e = _loss_scale_rule(coef) if f16 else 0
    with np.errstate(invalid="ignore", over="ignore"):
        coef = coef * np.float32(2.0 ** e)
        m = (mask.reshape(B, Hp * Wp) * coef).astype(np.float32)                 # mask 0 x inf = NaN, as on the device
    d = (x_rec - x).reshape(B, C, Hp, p, Wp, p).transpose(0, 2, 4, 1, 3, 5).reshape(B, Hp * Wp, C * p * p)
    mm = m[:, :, None]
    g = np.where(d > 0, mm, np.where(d < 0, -mm, np.float32(0)))
    g = np.where(mm != 0, g, np.float32(0))                                      # m == 0: the kernel writes +0
    dY = np.zeros((B, Hp * Wp + 1, C * p * p), np.float32)
    dY[:, 1:] = g
    return dY.reshape(B * (Hp * Wp + 1), C * p * p), e


def _run_mim_loss_bwd(eng, x, x_rec, mask, sums, gscale, B, H, W, dY, lscale):
    lib = vob._lib.load_library()
    check(lib.vitocm_mim_loss_bwd(eng, ptr(x), ptr(x_rec), ptr(mask), ptr(sums), ptr(gscale), B, H, W, ptr(dY), ptr(lscale), cur_stream()))
    torch.cuda.synchronize()


def _to16(a, prec):
    t = torch.from_numpy(a).cuda()
    return t.clamp(-65504, 65504).half() if prec == "fp16" else t.to(torch.bfloat16)   # fp16: saturating, like cvt.satfinite


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("C,p,B,H,W", [(3, 8, 1, 32, 32), (3, 8, 64, 32, 48), (1, 8, 5, 48, 32), (3, 16, 3, 64, 32), (3, 16, 1, 32, 48),
                                       (1, 8, 17, 224, 224)])
def test_mim_loss_backward(prec, C, p, B, H, W):
    """mim_loss_bwd_kernel bit-exact against the float32 restatement of its formula for gscale in {1, 2^-20, 2^20, 2^-120, 0, inf},
    within 16-bit rounding of float64 autograd of the model.py loss through PixelShuffle; fp16: the loss scale follows the rule of
    include/vitocm.h exactly (2^-120, and at C = 3 an all-zero mask at 2^112, hit the clamp at +-126)."""
    lib = vob._lib.load_library()
    eng = make_engine(patch=p, chans=C, precision=FP16 if prec == "fp16" else 0)
    dt = DT[prec]
    try:
        x, x_rec, mask, Y = _mim_inputs(B, C, H, W, p, 600 + B)
        Hp, Wp = H // p, W // p
        M, ldy = B * (Hp * Wp + 1), C * p * p
        cases = [(mask, g) for g in (1.0, 2.0 ** -20, 2.0 ** 20, 2.0 ** -120, 0.0, float("inf"))] + [(0 * mask, 2.0 ** 112)]
        for mk, gscale in cases:
            sums1 = float(mk.sum()) * p * p                               # sum of the pixel mask (model.py:75)
            sums = torch.tensor([1.0, sums1], dtype=torch.float64, device="cuda")
            gs = torch.tensor([gscale], device="cuda")
            dY = torch.full((M + PAD, ldy), float("nan"), device="cuda", dtype=dt)
            lscale = torch.full((2,), float("nan"), device="cuda")
            _run_mim_loss_bwd(eng, torch.from_numpy(x).cuda(), torch.from_numpy(x_rec).cuda(), torch.from_numpy(mk).cuda(), sums, gs, B, H, W,
                              dY, lscale)
            _assert_nan(dY[M:], "pad rows of dY")
            ref32, e = _mim_kernel_numpy(x, x_rec, mk, sums1, gscale, C, p, prec == "fp16")
            want = _to16(ref32, prec)
            got = dY[:M]
            nan_w, nan_g = torch.isnan(want.float()), torch.isnan(got.float())
            assert torch.equal(nan_w, nan_g), gscale
            assert torch.equal(got.view(torch.int16)[~nan_g], want.view(torch.int16)[~nan_w]), f"dY differs from the kernel formula (gscale {gscale})"
            if prec == "fp16":
                assert lscale.tolist() == [2.0 ** e, 2.0 ** -e], (gscale, lscale.tolist(), e)
            else:
                assert torch.isnan(lscale).all(), "bf16 engines do not write the loss scale"
            if gscale in (1.0, 2.0 ** -20, 2.0 ** 20) and mk is mask:
                # float64 autograd of loss = sum |x - PixelShuffle(Y)| mask_up / (sum mask_up + 1e-5) / C
                Y64 = torch.from_numpy(Y).double().cuda().requires_grad_(True)
                rec = torch.nn.functional.pixel_shuffle(Y64, p)
                mup = torch.from_numpy(mk).double().cuda().reshape(B, 1, Hp, Wp).repeat_interleave(p, 2).repeat_interleave(p, 3)
                loss = ((torch.from_numpy(x).double().cuda() - rec).abs() * mup).sum() / (mup.sum() + 1e-5) / C
                (loss * gscale).backward()
                ref = torch.zeros(B, Hp * Wp + 1, ldy, dtype=torch.float64, device="cuda")
                ref[:, 1:] = Y64.grad.reshape(B, ldy, Hp * Wp).transpose(1, 2) * 2.0 ** e
                ref = ref.reshape(M, ldy)
                g64 = got.double()
                bound = 0.5 * ulp16(torch.maximum(g64.abs(), ref.abs()), prec) + 4 * EPS24 * ref.abs()
                _assert_within(g64, ref, bound, f"dY vs autograd (gscale {gscale})")
    finally:
        lib.vitocm_destroy(eng)


def test_mim_loss_backward_refuses_fp32_parity_engines():
    lib = vob._lib.load_library()
    eng = make_engine(precision=1)
    try:
        with pytest.raises(vob.VitocmError, match="16-bit engines"):
            check(lib.vitocm_mim_loss_bwd(eng, None, None, None, None, None, 1, 32, 32, None, None, cur_stream()))
    finally:
        lib.vitocm_destroy(eng)


# ------------------------------------------------------------------------------------------------------------ clip and AdamW
@pytest.mark.parametrize("n", [100003, 4, 7])
@pytest.mark.parametrize("max_norm", [1e-2, 1e6])
def test_grad_clip(n, max_norm):
    """g <- g min(1, max_norm / (sqrt(sumsq) + 1e-6)) in place, the coefficient in float32 as the kernel forms it; the n % 4 tail too"""
    lib = vob._lib.load_library()
    g0 = _rand((n,), 700 + n, 0.3)
    g = g0.clone()
    ss = torch.zeros(1, dtype=torch.float64, device="cuda")
    check(lib.vitocm_grad_sumsq(ptr(g), n, ptr(ss), cur_stream()))
    check(lib.vitocm_grad_clip(ptr(g), n, max_norm, ptr(ss), cur_stream()))
    torch.cuda.synchronize()
    ref_ss = g0.double().pow(2).sum().item()
    assert abs(ss.item() - ref_ss) <= 1e-6 * ref_ss
    c = np.float32(max_norm) / (np.float32(math.sqrt(ss.item())) + np.float32(1e-6))
    want = (g0.cpu() * torch.tensor(float(c))) if c < 1 else g0.cpu()
    assert torch.equal(g.cpu(), want)
    assert (c < 1) == (max_norm < 1), "both sides of max_norm are covered"


@pytest.mark.parametrize("grad_scale,max_norm,with_sumsq", [(0.25, 1.0, True), (0.5, 0.0, True), (2.0, 5.0, False), (0.125, 1e6, True)])
def test_adamw_grad_scale_and_clip_modes(grad_scale, max_norm, with_sumsq):
    """vitocm_adamw_step with grad_scale != 1: g <- g grad_scale min(1, max_norm / (sqrt(sumsq) grad_scale + 1e-6)), no clipping for
    max_norm <= 0 or sumsq NULL; then AdamW with decoupled weight decay per element, three steps, against float64."""
    lib = vob._lib.load_library()
    n = 100003
    # the hyper-parameters as the kernel receives them (float32): 1 - f32(0.999) differs from 0.001 by 1.3e-5 relative
    lr, b1, b2, eps, wd = (float(np.float32(h)) for h in (5e-4, 0.9, 0.999, 1e-8, 0.05))
    p = _rand((n,), 800)
    m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    decay = (torch.arange(n, device="cuda") % 3 != 0).to(torch.uint8)
    P, Mm, V = p.double(), m.double(), v.double()
    Mabs = Mm.clone()                                  # the moment of |g|: what m's fp32 roundings scale with
    ss = torch.zeros(1, dtype=torch.float64, device="cuda")
    clipped = False
    for step in range(1, 4):
        g0 = _rand((n,), 810 + step, 0.01 * step)
        g = g0.clone()
        check(lib.vitocm_grad_sumsq(ptr(g), n, ptr(ss), cur_stream()))
        check(lib.vitocm_adamw_step(ptr(p), ptr(g), ptr(m), ptr(v), ptr(decay), n, lr, b1, b2, eps, wd, step, max_norm, grad_scale,
                                    ptr(ss) if with_sumsq else None, cur_stream()))
        torch.cuda.synchronize()
        coef = grad_scale
        if max_norm > 0 and with_sumsq:
            c = max_norm / (math.sqrt(ss.item()) * grad_scale + 1e-6)
            clipped |= c < 1
            coef *= min(1.0, c)
        G = g0.double() * coef
        P = torch.where(decay.bool(), P * (1 - lr * wd), P)
        Mm = b1 * Mm + (1 - b1) * G
        Mabs = b1 * Mabs + (1 - b1) * G.abs()
        V = b2 * V + (1 - b2) * G * G
        P = P - (lr / (1 - b1 ** step)) * Mm / (V.sqrt() / math.sqrt(1 - b2 ** step) + eps)
        # g written back scaled (and clipped): the float32 coefficient carries a few roundings
        _assert_within(g.double(), G, 16 * EPS24 * G.abs(), "g")
        _assert_within(m.double(), Mm, 16 * step * EPS24 * Mabs, "m")
        _assert_within(v.double(), V, 16 * step * EPS24 * V, "v")
        _assert_within(p.double(), P, 16 * EPS24 * P.abs() + 1e-4 * lr, "p")
    assert clipped == (grad_scale == 0.25), "the clipping case clips, the others do not"
