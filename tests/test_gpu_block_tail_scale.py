"""GPU (B200): the block-tail kernel (csrc/block_tail_sm100.cuh) element by element against the rounding-faithful float64 reference of
tests/block_half_oracle.py, in every form run_block_tail accepts (plain or folded LayerNorm affine x {XN out, next QKV out, neither}), at
the launch sizes the benchmark runs: 1 225 tiles of 785 rows (961 625 rows, 3 757 items over 74 CTA pairs, staggered, a ragged last item
of 89 rows whose second CTA has no live row) and a full chunk of 2 048 tiles (1 607 680 rows, more than 2^31 bytes of fp32 X).

Every launch writes into buffers with guard bands: NaN rows after M in X, XN and QKV, NaN columns beyond D of XN's pitch and beyond 3D
of QKV's, and CTX is read through a wider pitch whose extra columns hold NaN; all guards must stay NaN.  Large launches are relaunched
on sub-ranges of their rows (unstaggered launches of at most 74 items, one staggered launch, starts at multiples of 128 rows and at an
odd row): X, XN and QKV must be bit-identical to the whole launch -- no row may depend on its pair, its place in the item or the stagger.
Every row of every launch is checked (the float64 reference of 1.6 M rows takes seconds on the device).

Pinned fractions (16-bit outputs whose reference interval is one value) of the probe operands: the fraction is a property of the
reference alone (it does not look at the kernel's output).  At D = 384 / Hd = 1536 it is 0.77 (bf16) and 0.42 (fp16) for XN and QKV,
at D = 128 / Hd = 512 0.77 / 0.43, at D = 128 / Hd = 128 0.88 - 0.90 / 0.63 - 0.68 (800 rows, every form).  Growth of the windows
compounds: each stage's window feeds the next through the unpinned 16-bit values, so scaling every window by 1.5 leaves 0.41 - 0.44
(bf16) and 0.02 - 0.05 (fp16) at Hd >= 512 and 0.69 - 0.72 / 0.24 - 0.26 at Hd = 128, and scaling by 2 leaves 0.10 - 0.15 / 0.00 at
Hd >= 512 and 0.45 - 0.47 / 0.04 at Hd = 128.  The floors PIN_FLOOR (0.6 bf16, 0.3 fp16) sit below every measured fraction and above
what windows 1.5 times as wide would leave at Hd >= 512 (and twice as wide at Hd = 128), so the windows cannot quietly grow until the
check has no teeth."""
import time

import pytest
import torch

import block_half_oracle as BO
import vitocm_b200 as vob
from gpu_util import make_engine
from vitocm_b200._lib import check, cur_stream, ptr

pytestmark = pytest.mark.gpu

GUARD_ROWS, GUARD_COLS = 64, 64
PIN_FLOOR = {"bf16": 0.6, "fp16": 0.3}
FORMS = [(folded, nxt) for folded in (False, True) for nxt in (None, "xn", "qkv")]


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


@pytest.fixture(scope="module")
def engines():
    lib = vob._lib.load_library()
    e = {"bf16": make_engine(precision=0), "fp16": make_engine(precision=2)}
    yield e
    for h in e.values():
        lib.vitocm_destroy(h)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def tail_plan(M, D, Hd, with_qkv, sms):
    """run_block_tail's dispatch (vitocm_api.cu): work items of 256 rows over sms / 2 CTA pairs, start stagger in SM clocks"""
    items = -(-M // BO.ITEM_ROWS)
    pairs = sms // 2
    r, rounds = items % pairs, -(-items // pairs)
    late = (r - 1 if r > 0 else pairs - 1) / pairs
    work = D * (D + 2.0 * Hd + (3.0 * D if with_qkv else 0.0))
    stagger = int(105000.0 * work / (384.0 * (384.0 + 3072.0 + 1152.0))) if items > pairs and late <= 0.04 * rounds else 0
    return {"items": items, "pairs": pairs, "items_per_pair": rounds, "stagger_clk": stagger, "ragged_rows": M - (items - 1) * BO.ITEM_ROWS}


class Launch:
    """one launch's buffers with guard bands"""

    def __init__(self, o, prec, folded, nxt, M, D, Hd):
        self.o, self.prec, self.folded, self.nxt, self.M, self.D, self.Hd = o, prec, folded, nxt, M, D, Hd
        dt = BO.DT[prec]
        self.dt = dt
        self.ctx = torch.full((M, D + GUARD_COLS), float("nan"), device="cuda", dtype=dt)
        self.ctx[:, :D] = o["ctx"]
        self.w = {k: o[k].to(dt).contiguous() for k in ("Wp", "W1", "W2", "Wq")}
        self.v = {k: o[k].float().contiguous() for k in ("bp", "g2", "be2", "b1", "b2", "gn", "ben", "bq")}

    def run(self, eng, r0=0, r1=None):
        """launch on rows [r0, r1): returns (X, XN, QKV) buffers with their guard rows / columns"""
        r1 = self.M if r1 is None else r1
        n, D = r1 - r0, self.D
        X = torch.full((n + GUARD_ROWS, D), float("nan"), device="cuda")
        X[:n] = self.o["X0"][r0:r1]
        XN = torch.full((n + GUARD_ROWS, D + GUARD_COLS), float("nan"), device="cuda", dtype=self.dt)
        QKV = torch.full((n + GUARD_ROWS, 3 * D + GUARD_COLS), float("nan"), device="cuda", dtype=self.dt) if self.nxt == "qkv" else None
        lib = vob._lib.load_library()
        fn = lib.vitocm_block_tail_folded if self.folded else lib.vitocm_block_tail
        w, v, ln = self.w, self.v, self.nxt is not None
        q = self.nxt == "qkv"
        check(fn(eng, ptr(self.ctx[r0:r1]), self.ctx.stride(0), ptr(w["Wp"]), D, ptr(v["bp"]), ptr(v["g2"]), ptr(v["be2"]), ptr(w["W1"]), D,
                 ptr(w["W2"]), self.Hd, n, D, self.Hd, ptr(v["b1"]), ptr(v["b2"]), ptr(X), ptr(v["gn"]) if ln else None, ptr(v["ben"]) if ln else None,
                 ptr(XN), XN.stride(0), ptr(w["Wq"]) if q else None, D, ptr(v["bq"]) if q else None, ptr(QKV) if q else None,
                 QKV.stride(0) if q else 0, None, cur_stream()))
        torch.cuda.synchronize()
        return X, XN, QKV

    def check_guards(self, X, XN, QKV, n):
        D = self.D
        assert torch.isnan(X[n:]).all(), "X: a guard row after M was written"
        if self.nxt == "xn":
            assert torch.isnan(XN[n:].float()).all() and torch.isnan(XN[:n, D:].float()).all(), "XN: a guard row / column was written"
        else:
            assert torch.isnan(XN.float()).all(), "XN written although the form does not write it"
        if QKV is not None:
            assert torch.isnan(QKV[n:].float()).all() and torch.isnan(QKV[:n, 3 * D:].float()).all(), "QKV: a guard row / column was written"

    def outputs(self, X, XN, QKV, n):
        got = {"x": X[:n]}
        if self.nxt == "xn":
            got["xn"] = XN[:n, :self.D]
        if self.nxt == "qkv":
            got["qkv"] = QKV[:n, :3 * self.D]
        return got


def run_case(engines, kind, prec, D, Hd, M, folded, nxt, seed, expect, pin_floor=True, sub_launches=(), **recipe):
    """one launch against the reference on every row; expect = (items per pair, stagger clocks) of the dispatch on a B200"""
    t0 = time.time()
    plan = tail_plan(M, D, Hd, nxt == "qkv", _sms())
    if _sms() == 148:
        assert (plan["items_per_pair"], plan["stagger_clk"]) == expect, (M, D, Hd, nxt, plan)
    o = BO.fold(BO.operands(kind, prec, D, Hd, M, seed, device="cuda", **recipe), prec, folded, folded and nxt == "qkv")
    L = Launch(o, prec, folded, nxt, M, D, Hd)
    X, XN, QKV = L.run(engines[prec])
    L.check_guards(X, XN, QKV, M)
    got = L.outputs(X, XN, QKV, M)
    for k, t in got.items():
        assert torch.isfinite(t.float()).all(), f"{k}: non-finite output"
    ops = BO.reference(o, prec, folded, folded, nxt)
    rep = BO.check_launch(ops, got)
    line = (f"{kind} {prec} D={D} Hd={Hd} M={M} {'folded' if folded else 'plain'} next={nxt}: items/pair {plan['items_per_pair']} "
            f"stagger {plan['stagger_clk']} clk, every row checked; {rep}")
    assert rep.ok(), line
    if pin_floor:
        for k in ("xn", "qkv"):
            if k in got:
                assert rep.pinned_fraction(k) >= PIN_FLOOR[prec], f"{k}: pinned fraction {rep.pinned_fraction(k):.3f} < {PIN_FLOOR[prec]}: {line}"
    for r0, r1 in sub_launches:
        sp = tail_plan(r1 - r0, D, Hd, nxt == "qkv", _sms())
        Xs, XNs, QKVs = L.run(engines[prec], r0, r1)
        L.check_guards(Xs, XNs, QKVs, r1 - r0)
        for k, t in L.outputs(Xs, XNs, QKVs, r1 - r0).items():
            whole = got[k][r0:r1]
            same = t.contiguous().view(torch.int32 if k == "x" else torch.int16) == whole.contiguous().view(torch.int32 if k == "x" else torch.int16)
            if not bool(same.all()):
                i, j = (~same).nonzero()[0].tolist()
                pytest.fail(f"{k}: rows [{r0}, {r1}) relaunched (stagger {sp['stagger_clk']}) differ from the whole launch, first at row "
                            f"{r0 + i} column {j}: {float(t[i, j])} vs {float(whole[i, j])}")
    if sub_launches:
        line += f"; sub-batches bit-identical ({len(sub_launches)} relaunches)"
    print(f"\n{line}  [{time.time() - t0:.1f} s]")
    return rep


# ------------------------------------------------------------------------------------------------------------ forms and widths
@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("D,Hd", [(384, 1536), (128, 128), (128, 384), (128, 512)])
def test_block_tail_forms(engines, prec, D, Hd):
    """every form on the probe operands (pinned-fraction floor) and on dense ones, ragged launch of 3 items + 17 rows"""
    M = 3 * 256 + 17
    for folded, nxt in FORMS:
        run_case(engines, "probe", prec, D, Hd, M, folded, nxt, 10 + D + Hd, (1, 0))
        run_case(engines, "dense", prec, D, Hd, M, folded, nxt, 20 + D + Hd, (1, 0), pin_floor=False)


# ------------------------------------------------------------------------------------------------------------ launch sizes
# (M, expected items per pair, stagger clocks) of ViT-S launches at D = 384, Hd = 1536 with the next QKV (sms = 148)
SIZES = [(1, 1, 0), (257, 1, 0), (785, 1, 0), (137375, 8, 105000), (961625, 51, 105000), (1607680, 85, 105000)]
SUBS = {137375: [(0, 74 * 256), (128 * 37, 128 * 37 + 9000), (12345, 12345 + 7777), (768, 768 + 370 * 256 + 100)],
        961625: [(961625 - 74 * 256, 961625), (128 * 5001, 128 * 5001 + 15000), (400001, 400001 + 5555), (256 * 1000, 256 * 1000 + 370 * 256 + 100)],
        1607680: [(1607680 - 74 * 256, 1607680), (2 ** 31 // (4 * 384) - 4000, 2 ** 31 // (4 * 384) + 4000)]}


@pytest.mark.parametrize("M,per_pair,stagger", SIZES)
def test_block_tail_launch_sizes_fp16_folded_qkv(engines, M, per_pair, stagger):
    """the form the forward runs on fp16 engines, up to a full chunk; the dispatch mirror pins which launches are staggered"""
    plan = tail_plan(M, 384, 1536, True, _sms())
    if _sms() == 148:
        if M == 961625:
            assert plan["items"] == 3757 and plan["ragged_rows"] == 89     # the second CTA of the last item has no live row
    subs = SUBS.get(M, ())
    if _sms() == 148:
        for r0, r1 in subs:   # the relaunches: unstaggered launches of <= 74 items, one staggered one (371 items: r = 1)
            sp = tail_plan(r1 - r0, 384, 1536, True, 148)
            assert (sp["stagger_clk"] > 0) == (sp["items"] > 74), (r0, r1, sp)
    run_case(engines, "probe", "fp16", 384, 1536, M, True, "qkv", 30, (per_pair, stagger), sub_launches=subs)


# without the QKV chunks an item carries 3/4 of the work, and the stagger scales with it: 78 750 clocks
@pytest.mark.parametrize("M,prec,folded,nxt,per_pair,stagger", [(137375, "bf16", True, "qkv", 8, 105000), (961625, "bf16", False, "xn", 51, 78750),
                                                                (961625, "fp16", False, None, 51, 78750), (137375, "fp16", False, "qkv", 8, 105000),
                                                                (1607680, "bf16", True, "qkv", 85, 105000), (137375, "bf16", True, "xn", 8, 78750)])
def test_block_tail_launch_sizes_other_forms(engines, M, prec, folded, nxt, per_pair, stagger):
    run_case(engines, "probe", prec, 384, 1536, M, folded, nxt, 40, (per_pair, stagger),
             sub_launches=SUBS[137375][-1:] if M == 137375 else ())


# ------------------------------------------------------------------------------------------------------------ edges
@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("D,Hd", [(384, 1536), (128, 512)])
def test_block_tail_constant_rows(engines, prec, D, Hd):
    """CTX row 0, bias_p 0, X row = 0, 1.5 or -250 on every 7th row: the kernel's mean is exactly c and its M2 exactly 0 (every partial
    sum exact), so norm2's rows are the exact residual of fma(c, rstd, -c rstd) -- the reference gives them no statistics window"""
    M = 4 * 256 + 100
    o = BO.operands("probe", prec, D, Hd, M, 50, device="cuda", const_rows=True)
    ops = BO.reference(o, prec, False, False, None)
    assert int(ops.rows(torch.arange(M, device="cuda"))["exact_rows"].sum()) == len(range(3, M, 7)), "every constant row has exact statistics"
    for folded, nxt in FORMS:
        run_case(engines, "probe", prec, D, Hd, M, folded, nxt, 50, (1, 0), pin_floor=False, const_rows=True)


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("kind", ["probe", "dense"])
def test_block_tail_large_means(engines, prec, kind):
    """rows offset by 20 and -150 standard deviations: the fp32 statistics' error, amplified by rstd, stays inside its window"""
    for folded, nxt in ((False, "xn"), (True, "qkv"), (False, "qkv")):
        run_case(engines, kind, prec, 384, 1536, 1100, folded, nxt, 60, (1, 0), pin_floor=False, large_means=True)
