"""CPU: the block-half checker (tests/block_half_oracle.py) has teeth.  An fp32 emulation of the block-tail kernel -- round-to-nearest
16-bit stores, its own summation order, the engine's own sigmoid-form GELU (within the documented error of erf GELU) -- passes in every
form; each plausible slip of a later optimisation of the kernel, emulated one at a time, fails.

Operand sets (block_half_oracle.operands).  "dense": random operands as a block carries them, with rows far from zero (acceptance
only: the 16-bit ambiguity of one stage spreads through the next dense product, so its windows are loose).  "probe": few non-zeros per
weight row, so that each output exposes single hidden values -- the set every slip is tried on.  "const": the probe set with the rows the
kernel must normalise exactly (CTX row 0, bias_p 0, X row constant at 0, 1.5 or -250)."""
import math

import pytest
import torch

import block_half_oracle as BO

M_ROWS = 600          # two full work items and a ragged one of 88 rows
SHAPES = [(128, 256), (384, 1536)]


def _operands(kind, prec, D, Hd, seed):
    """dense: with rows far from zero; probe; const: probe with the exactly normalised constant rows (bias_p 0)"""
    return BO.operands("dense" if kind == "dense" else "probe", prec, D, Hd, M_ROWS, seed, const_rows=kind == "const",
                       large_means=kind == "dense")


fold = BO.fold
oracle_ops = BO.reference


# ------------------------------------------------------------------------------------------------------------ fp32 emulation
def _fma(a, b, c):
    return (a.double() * b.double() + c.double()).float()


def gelu_sigmoid3(x):
    """the three-coefficient form of bf16 engines (gemm_sm100.cuh), in float64"""
    u = torch.clamp(x * x, max=100.0)
    w = (0.0010142630596 * u - 0.1067757240) * u - 2.3011213394
    return x / (1.0 + torch.pow(2.0, x * w))


def gelu_sigmoid5(x):
    """the five-coefficient form of fp16 engines (gemm_sm100.cuh), in float64"""
    u = x * x
    w = (((-3.2290010e-06 * u + 8.8238336e-05) * u + 3.6027357e-04) * u - 0.10522669) * u - 2.3020453
    return x / (1.0 + torch.pow(2.0, x * w))


def _store16(v32, prec, rz):
    q = BO.rn16(v32.double(), prec)
    if not rz:
        return q
    qd, vd = q.double(), v32.double()
    away = qd.abs() > vd.abs()
    return torch.where(away, qd - torch.sign(vd) * BO.ulp16(vd, prec), qd).to(q.dtype)


def _ln32(y, gamma, beta, eps, const_m2=None):
    mean = y.mean(1, keepdim=True)
    var = ((y - mean) ** 2).mean(1, keepdim=True)
    if const_m2 is not None:                                            # mutation: constant rows normalised with M2 != 0
        var = torch.where(const_m2[:, None], BO.ulp32(mean.double()).float() ** 2 + var, var)
    r = torch.rsqrt(var + torch.tensor(eps, dtype=torch.float32))
    n = _fma(y, r, -mean * r)
    return n if gamma is None else _fma(n, gamma, beta)


def emulate(o, prec, fold2, foldn, nxt, mut=()):
    """the block-tail kernel's arithmetic in fp32 (torch's summation orders), 16-bit stores where the kernel has them"""
    f = lambda k: o[k].float()
    bp = torch.roll(f("bp"), -32) if "bias_p_shift" in mut else f("bp")
    y = (f("X0") + bp) + f("ctx") @ f("Wp").T
    const = (y == y[:, :1]).all(1) if "const_m2" in mut else None
    n2 = _ln32(y, f("g2") if (not fold2 or "gamma_twice" in mut) else None, f("be2"), 1e-6, const)
    u_n2 = _store16(n2, prec, False)
    pre = u_n2.float() @ f("W1").T + f("b1")
    form = gelu_sigmoid3 if (prec == "bf16" or "gelu3_fp16" in mut) else gelu_sigmoid5
    h = _store16(form(pre.double()).float(), prec, "hidden_rz" in mut)
    acc = h.float() @ f("W2").T
    out = y + acc
    b2 = f("b2").expand_as(out).clone()
    if "b2_box" in mut:
        b2[ITEM1 + 32:ITEM1 + 64, 32:64] = 0
    x = out + b2
    got = {"x": x}
    if nxt is not None:
        plain = nxt == "xn" or not foldn or "xn_plain_in_folded" in mut
        xn = _ln32(x, f("gn") if plain else None, f("ben"), 1e-6)
        u_xn = _store16(xn, prec, "xn_rz" in mut)
        if nxt == "xn":
            got["xn"] = u_xn
        else:
            got["qkv"] = _store16(u_xn.float() @ f("Wq").T + f("bq"), prec, False)
    if "stale_box" in mut:                                              # one 32-row box of item 1 holds item 0's rows
        for k in got:
            got[k] = got[k].clone()
            got[k][ITEM1 + 64:ITEM1 + 96] = got[k][64:96]
    return got


ITEM1 = BO.ITEM_ROWS


FORMS = [(fold2, foldn, nxt) for fold2 in (False, True) for nxt, foldn in ((None, False), ("xn", False), ("qkv", False), ("qkv", True))]


@pytest.mark.parametrize("kind", ["dense", "probe", "const"])
@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("D,Hd", SHAPES)
def test_emulated_kernel_is_accepted(kind, prec, D, Hd):
    """every form run_block_tail accepts: folded or plain norm2 x {XN out, QKV out (plain or folded next norm1), neither}"""
    o0 = _operands(kind, prec, D, Hd, 7)
    for fold2, foldn, nxt in FORMS:
        o = fold(o0, prec, fold2, foldn)
        got = emulate(o, prec, fold2, foldn, nxt)
        rep = BO.check_launch(oracle_ops(o, prec, fold2, foldn, nxt), got)
        assert rep.ok(), f"fold2={fold2} foldn={foldn} next={nxt}: {rep}"
        print(f"\n{kind} {prec} D={D} Hd={Hd} fold2={fold2} foldn={foldn} next={nxt}: {rep}")


# (name, operand set, precisions, form): the form in which the slip exists; the probe operands, where each output exposes single values
MUTATIONS = [
    ("xn_rz", "probe", ("bf16", "fp16"), (False, False, "xn")),              # RZ instead of RN in the XN store
    ("hidden_rz", "probe", ("bf16", "fp16"), (True, True, "qkv")),           # RZ in the hidden-activation store
    ("gelu3_fp16", "probe", ("fp16",), (True, True, "qkv")),                 # the three-coefficient GELU on an fp16 engine
    ("gamma_twice", "probe", ("bf16", "fp16"), (True, True, "qkv")),         # gamma2 applied on top of the folded W1
    ("xn_plain_in_folded", "probe", ("bf16", "fp16"), (True, True, "qkv")),  # the plain XN affine in the folded-QKV form
    ("b2_box", "probe", ("bf16", "fp16"), (True, False, "xn")),              # b2 missing from one 32-column box
    ("bias_p_shift", "probe", ("bf16", "fp16"), (True, True, "qkv")),        # bias_p read 32 columns off
    ("stale_box", "probe", ("bf16", "fp16"), (True, True, "qkv")),           # one 32-row box of an item holds another item's rows
    ("const_m2", "const", ("bf16", "fp16"), (True, True, "qkv")),            # a constant row normalised with M2 != 0
]


@pytest.mark.parametrize("D,Hd", SHAPES)
@pytest.mark.parametrize("name,kind,precs,form", MUTATIONS, ids=[m[0] for m in MUTATIONS])
def test_mutation_is_rejected(name, kind, precs, form, D, Hd):
    fold2, foldn, nxt = form
    for prec in precs:
        o = fold(_operands(kind, prec, D, Hd, 11), prec, fold2, foldn)
        ops = oracle_ops(o, prec, fold2, foldn, nxt)
        assert BO.check_launch(ops, emulate(o, prec, fold2, foldn, nxt)).ok(), "the unmutated emulation must pass"
        rep = BO.check_launch(ops, emulate(o, prec, fold2, foldn, nxt, (name,)))
        assert not rep.ok(), f"{name} ({prec}, D={D}) passed the checker: {rep}"
        print(f"\n{name} {prec} D={D}: rejected: {rep}")


def test_rounding_helpers():
    """RN16 saturates like cvt.rn.satfinite and keeps subnormals; ulp16 / ulp32 give the subnormal spacing below the normal range"""
    x = torch.tensor([70000.0, -1e9, 65519.0, 2.0 ** -20, 0.0], dtype=torch.float64)
    assert BO.rn16(x, "fp16").double().tolist() == [65504.0, -65504.0, 65504.0, 2.0 ** -20, 0.0]
    assert BO.ulp16(torch.tensor([2.0 ** -20, 1.0], dtype=torch.float64), "fp16").tolist() == [2.0 ** -24, 2.0 ** -10]
    assert BO.ulp16(torch.tensor([1.0], dtype=torch.float64), "bf16").tolist() == [2.0 ** -7]
    assert BO.ulp32(torch.tensor([0.0, 1.0], dtype=torch.float64)).tolist() == [2.0 ** -149, 2.0 ** -23]
    assert abs(BO.gelu64(torch.tensor([1.0], dtype=torch.float64)).item() - 0.8413447460685429) < 1e-15
    t = torch.linspace(-12, 12, 200001, dtype=torch.float64)
    for form, prec, documented in ((gelu_sigmoid3, "bf16", 2.5e-5), (gelu_sigmoid5, "fp16", 3.0e-6)):   # the emulated forms, their error
        err = (form(t) - BO.gelu64(t)).abs().max().item()
        assert 0.9 * documented <= err <= BO.GELU_ERR[prec], (prec, err)
    assert math.isclose(BO.KS * BO.EPS24, 32 * 2.0 ** -24)
