"""Rounding-faithful float64 reference of the second half of a transformer block, as the block-tail kernel
(csrc/block_tail_sm100.cuh) computes it (Operands), and of the stages of the unfused path taken one by one (stage_*), with a
per-element window at every stage.

Given the exact 16-bit and fp32 operands a kernel reads, the reference evaluates

    y   = X + bias_p + CTX . Wp^T                           proj + residual                    fp32
    n2  = LayerNorm(y; ln2)  (folded: (y - mean) rstd)       norm2                              16 bit
    h   = gelu(n2 . W1^T + b1)                               fc1 + GELU                         16 bit
    x   = y + h . W2^T + b2                                  fc2 + residual                     fp32 (output X)
    xn  = LayerNorm(x; next norm1)  (folded: (x - mean) rstd)                                   16 bit (output XN, or kept)
    qkv = xn . Wqkv^T + bqkv                                 the next block's QKV projection    16 bit (output QKV)

in float64 and rounds to 16 bits at exactly the points where the kernels do.  Every stage carries a window w: a bound on how far the
kernel's fp32 value at that point can lie from the float64 value v.  It is built from

* fp32 accumulation: (K + 2) 2^-24 sum |a| |b| over the K products of an output (K counts the non-zero products only: adding an exact
  zero does not round), the model of tests/test_gpu_train_epilogues.py;
* fp32 LayerNorm statistics (exact (mean, M2) per 32 values, Chan's combination): every value goes through at most KS = 32 fp32
  roundings (8 sequential adds per accumulator, 2 tree adds, the scaling, two Chan steps of 4 operations, 5 in the cross-warp
  combination), so mean and M2 carry KS 2^-24 relative to sum |y| -- an error that (y - mean) rstd amplifies by rstd, which is why the
  window scales with rstd mean |y| (rows far from zero); rsqrtf adds 2 ulp (2^-22 relative);
* the documented maximum error of the engine's GELU form (gemm_sm100.cuh): 2.5e-5 for the three-coefficient form of bf16 engines,
  3.0e-6 for the five-coefficient form of fp16 engines (2.6e-5 / 3.1e-6 here: the exact maxima are 2.52e-5 / 3.04e-6), plus 2^-21 |x| for the approximate ex2 / rcp;

and, on top, the propagated deviation of the upstream 16-bit values as a float64 GEMM of absolute values (|W| @ dev).  At a 16-bit
point the reference keeps u = RN16(v) and records dev = max(RN16(v + w) - u, u - RN16(v - w)) -- 0 wherever the rounding is
unambiguous.  Each window is at least one fp32 ulp of v (the kernel's value is an fp32 number).  First-order terms only: the
second-order ones are below 2^-40 relative at these magnitudes.

Rows whose statistics are exact: a row of y that is exactly constant (CTX row 0 and bias_p 0 make y = X exactly) with a value of at
most 15 significant bits has every partial sum of the statistics exact for D <= 384 (32 c and 384 c need at most 9 more bits), so the
kernel's mean is c and its M2 exactly 0; rstd = rsqrtf(eps) and (x - mean) rstd = fma(c, rstd, -c rstd) is the exact rounding residual of
c rstd.  Those rows get no statistics window at all: only the spread of that residual over the 2-ulp candidates of rsqrtf(eps).  A
kernel that forms a non-zero M2 or an inexact mean on them lands elsewhere.

The checks: a 16-bit output must satisfy RN16(v - w) <= got <= RN16(v + w) (where that interval is one value the output is pinned bit
for bit); an fp32 output must satisfy |got - v| <= w.  Each check reports the fraction of 16-bit outputs that are pinned and the worst
error / window with its (item, row, column); items are the kernel's 256-row work items.

Operand recipes (`operands`): "dense" -- random operands as a block carries them; there the 16-bit ambiguity of one stage spreads
through |W| @ dev of the next dense product, so the windows of X / XN / QKV are loose and few 16-bit outputs are pinned.  "probe" --
Wp, W1, W2 and Wqkv hold few non-zeros per row (X column i reads the hidden units i, i + D, ..., hidden unit j reads normalised column
j mod D, QKV column k reads XN column k mod D), so every accumulation is exact or nearly so, most 16-bit points are pinned, and each
output element exposes single hidden values: a slip of a fraction of a 16-bit ulp in the hidden store or in the GELU shows in X.  The
pre-activations a n + b1 with |a| up to 4 reach both GELU tails.

The unfused path (LayerNorm kernel, QKV GEMM, proj GEMM with TMA reduce-add into X, LayerNorm, fc1 GEMM with GELU, fc2 GEMM with
reduce-add) rounds in its own order -- the reduce-add forms X + RN(acc + bias), not (X + bias) + acc -- so its stages have their own
functions, each on the exact inputs the stage reads: stage_linear (acc + bias, to 16 bits or fp32), stage_gelu, stage_reduce_add and
stage_layernorm (vit_kernels.cuh, one warp per row: a value goes through at most 2 + D / 128 + 5 + 1 <= 14 fp32 roundings of the
statistics at D <= 1024, inside KS).

Importable without a GPU or pytest (numpy / torch only); it runs on the operands' device, chunked over rows.
"""
import math

import torch

EPS24 = 2.0 ** -24
KS = 32                                   # fp32 roundings a value sees in the LayerNorm statistics (see above)
RSQRT_REL = 2.0 ** -22                    # rsqrtf: 2 ulp
# maximum |form - erf GELU| over the real line: the three-coefficient form reaches 2.52e-5 (documented as 2.5e-5), the five-coefficient
# one 3.04e-6 (documented as 3.0e-6)
GELU_ERR = {"bf16": 2.6e-5, "fp16": 3.1e-6}
GELU_APPROX_REL = 2.0 ** -21              # ex2.approx / rcp.approx of the sigmoid forms, relative to |x|
GELU_SLOPE = 1.13                         # max |gelu'|
MANT = {"bf16": 7, "fp16": 10}            # stored significand bits
EMIN = {"bf16": -126, "fp16": -14}        # exponent of the smallest normal value
DT = {"bf16": torch.bfloat16, "fp16": torch.float16}
FP16_MAX = 65504.0
ITEM_ROWS = 256                           # rows of one work item (a CTA pair's tile)


def ulp16(x, prec):
    """ulp of the 16-bit format at |x| (float64 tensor), subnormal spacing below the smallest normal"""
    _, ex = torch.frexp(x.abs())
    e = torch.where(x == 0, EMIN[prec], torch.clamp(ex.to(torch.float64) - 1, min=EMIN[prec]))
    return torch.pow(2.0, e - MANT[prec])


def ulp32(x):
    """ulp of fp32 at |x| (float64 tensor), subnormal spacing below 2^-126"""
    _, ex = torch.frexp(x.abs())
    e = torch.where(x == 0, -126, torch.clamp(ex.to(torch.float64) - 1, min=-126))
    return torch.pow(2.0, e - 23)


def gelu64(x):
    return 0.5 * x * (1.0 + torch.special.erf(x / math.sqrt(2.0)))


def rn16(x, prec):
    """round to nearest even into the 16-bit format (through fp32, as the kernels round their fp32 values); fp16 saturates at
    65504 like cvt.rn.satfinite.  Monotone, so RN16(v - w) <= RN16(k) <= RN16(v + w) for every fp32 k in [v - w, v + w]."""
    x32 = x.float()
    if prec == "fp16":
        return x32.clamp(-FP16_MAX, FP16_MAX).half()
    return x32.to(torch.bfloat16)


def _at16(v, w, prec):
    """a 16-bit point: u = RN16(v) (float64) and dev = how far the kernel's 16-bit value may lie from u"""
    u = rn16(v, prec).double()
    lo, hi = rn16(v - w, prec).double(), rn16(v + w, prec).double()
    return u, torch.maximum(hi - u, u - lo)


def _window(v, w):
    return torch.maximum(w, ulp32(v))


def _nnz(A, B):
    """non-zero products per output of A @ B^T (K where neither operand holds a zero)"""
    if bool((A != 0).all()) and bool((B != 0).all()):
        return float(A.shape[1])
    return (A != 0).double() @ (B != 0).double().T


def _linear(a, dev, W64, Wabs, Wnz, bias):
    """out = a . W^T + bias of 16-bit rows a (float64 values) whose kernel value may differ by dev: value and window"""
    v = a @ W64.T + bias
    mag = a.abs() @ Wabs.T + bias.abs()
    k = _nnz(a, Wnz) if Wnz is not None else float(W64.shape[1])
    return v, (k + 2.0) * EPS24 * mag + dev @ Wabs.T


def _layernorm(y, wy, gamma, beta, eps, exact_rows=None):
    """(y - mean) rstd [* gamma + beta] from fp32 rows y (float64 values, window wy) as the kernels form it:
    fma(y, rstd, -mean rstd), then fma(., gamma, beta) in the plain form (gamma None: folded)"""
    D = y.shape[1]
    mean = y.mean(1, keepdim=True)
    var = ((y - mean) ** 2).mean(1, keepdim=True)
    eps32 = float(torch.tensor(eps, dtype=torch.float32))
    r = 1.0 / torch.sqrt(var + eps32)
    nh = (y - mean) * r
    # the kernel's y is not the reference's y: its mean moves by at most mean(wy), its variance by 2 mean(|y - mean| wy)
    w = r * (wy + wy.mean(1, keepdim=True)) + nh.abs() * r * r * ((y - mean).abs() * wy).mean(1, keepdim=True)
    w = w + KS * EPS24 * (1.0 + r * y.abs().mean(1, keepdim=True)) * (1.0 + nh.abs()) + RSQRT_REL * nh.abs()
    if exact_rows is not None and bool(exact_rows.any()):
        # exact statistics (module docstring): mean = c, M2 = 0, rstd one of the 2-ulp candidates of rsqrtf(eps)
        r0 = torch.tensor(1.0 / math.sqrt(eps32), dtype=torch.float32, device=y.device)
        cands = [r0.double() + k * ulp32(r0.double()) for k in (-2, -1, 0, 1, 2)]
        c = y[:, :1]
        res = torch.stack([c * rk - (c * rk).float().double() for rk in cands])   # fma(c, r, RN(-c r)): exact residual
        lo, hi = res.min(0).values, res.max(0).values
        nh = torch.where(exact_rows[:, None], 0.5 * (lo + hi), nh)
        w = torch.where(exact_rows[:, None], 0.5 * (hi - lo), w)
        if gamma is not None:
            w = torch.where(exact_rows[:, None], w * gamma.abs(), w)
    if gamma is None:
        return nh, _window(nh, w)
    v = nh * gamma + beta
    w = gamma.abs() * w if exact_rows is None else torch.where(exact_rows[:, None], w, gamma.abs() * w)
    return v, _window(v, w + EPS24 * v.abs())


def _exact_stat_rows(y, wy):
    """rows whose fp32 statistics are exact (module docstring)"""
    c = y[:, :1]
    const = (y == c).all(1) & (wy.max(1).values == 0)
    m, _ = torch.frexp(c[:, 0].abs())
    few_bits = (m * 2.0 ** 15 == torch.round(m * 2.0 ** 15))
    return const & few_bits


class Operands:
    """The exact operands of one block half, float64 on their device.  16-bit tensors: ctx [M][D], Wp [D][D], W1 [Hd][D], W2 [D][Hd],
    Wq [3D][D]; fp32 vectors: bp, g2, be2, b1, b2, gn, ben, bq; X0 [M][D] fp32 (the residual rows before the launch).  fold2: W1 / b1
    already carry norm2's gamma / beta (g2, be2 unused); foldn: Wq / bq carry the next norm1's (gn, ben unused).  nxt: None, "xn" or
    "qkv"."""

    def __init__(self, prec, ctx, Wp, bp, X0, W1, b1, W2, b2, g2=None, be2=None, gn=None, ben=None, Wq=None, bq=None, eps=1e-6,
                 fold2=False, foldn=False, nxt=None):
        self.prec, self.eps, self.fold2, self.foldn, self.nxt = prec, eps, fold2, foldn, nxt
        d = lambda t: None if t is None else t.double()
        self.ctx, self.X0 = ctx, X0
        self.Wp, self.W1, self.W2, self.Wq = d(Wp), d(W1), d(W2), d(Wq)
        self.bp, self.b1, self.b2, self.bq = d(bp), d(b1), d(b2), d(bq)
        self.g2, self.be2, self.gn, self.ben = d(g2), d(be2), d(gn), d(ben)
        self.abs = {k: getattr(self, k).abs() for k in ("Wp", "W1", "W2", "Wq") if getattr(self, k) is not None}
        self.nz = {k: (getattr(self, k) if bool((getattr(self, k) == 0).any()) else None) for k in self.abs}

    def rows(self, idx):
        """reference values and windows of the rows idx (LongTensor) of one launch: dict of (v, w) and, at 16-bit points, (u, dev)"""
        ctx = self.ctx[idx].double()
        X0 = self.X0[idx].double()
        out = ctx @ self.Wp.T
        mag = ctx.abs() @ self.abs["Wp"].T
        k = _nnz(ctx, self.nz["Wp"]) if self.nz["Wp"] is not None else float(self.Wp.shape[1])
        t = X0 + self.bp
        y = t + out
        wy = (k + 2.0) * EPS24 * mag
        wy = wy + EPS24 * torch.where((X0 != 0) & (self.bp != 0), t.abs(), 0.0) + EPS24 * torch.where(mag != 0, y.abs(), 0.0)
        exact = _exact_stat_rows(y, wy)
        n2, wn2 = _layernorm(y, wy, None if self.fold2 else self.g2, None if self.fold2 else self.be2, self.eps, exact)
        u_n2, dev_n2 = _at16(n2, wn2, self.prec)
        pre, wpre = _linear(u_n2, dev_n2, self.W1, self.abs["W1"], self.nz["W1"], self.b1)
        h = gelu64(pre)
        wh = _window(h, GELU_ERR[self.prec] + GELU_APPROX_REL * pre.abs() + GELU_SLOPE * wpre)
        u_h, dev_h = _at16(h, wh, self.prec)
        acc = u_h @ self.W2.T
        mag2 = u_h.abs() @ self.abs["W2"].T
        k2 = _nnz(u_h, self.nz["W2"]) if self.nz["W2"] is not None else float(self.W2.shape[1])
        x = y + acc + self.b2
        wx = wy + (k2 + 2.0) * EPS24 * (mag2 + y.abs()) + dev_h @ self.abs["W2"].T + EPS24 * torch.where(self.b2 != 0, x.abs(), 0.0)
        res = {"x": (x, _window(x, wx)), "y": (y, _window(y, wy)), "n2": (u_n2, dev_n2), "h": (u_h, dev_h), "exact_rows": exact}
        if self.nxt is None:
            return res
        plain = self.nxt == "xn" or not self.foldn
        xn, wxn = _layernorm(x, res["x"][1], self.gn if plain else None, self.ben if plain else None, self.eps)
        res["xn"] = (xn, wxn)
        if self.nxt == "qkv":
            u_xn, dev_xn = _at16(xn, wxn, self.prec)
            q, wq = _linear(u_xn, dev_xn, self.Wq, self.abs["Wq"], self.nz["Wq"], self.bq)
            res["qkv"] = (q, _window(q, wq))
        return res


class Report:
    """worst error / window, pinned fraction and first failures per output, accumulated over chunks of rows"""

    def __init__(self):
        self.out = {}

    def add(self, name, rows, got, v, w, prec=None):
        got = got.double()
        if prec is None:                                    # fp32 output
            err = (got - v).abs()
            ratio = err / w
            bad = ~(err <= w)
            pinned = None
        else:
            lo, hi = rn16(v - w, prec).double(), rn16(v + w, prec).double()
            bad = ~((got >= lo) & (got <= hi))
            d = got - v
            span = torch.where(d >= 0, hi - v, v - lo)
            ratio = torch.where(d == 0, 0.0, d.abs() / span)
            pinned = (lo == hi)
        ratio = torch.where(torch.isnan(ratio), float("inf"), ratio)
        s = self.out.setdefault(name, {"n": 0, "pinned": 0, "bad": 0, "worst": -1.0, "at": None, "first_bad": None, "is16": prec is not None})
        s["n"] += got.numel()
        if pinned is not None:
            s["pinned"] += int(pinned.sum())
        nb = int(bad.sum())
        if nb and s["first_bad"] is None:
            i, j = bad.nonzero()[0].tolist()
            row = int(rows[i])
            s["first_bad"] = (row // ITEM_ROWS, row % ITEM_ROWS, j, float(got[i, j]), float(v[i, j]), float(w[i, j]))
        s["bad"] += nb
        m = float(ratio.max())
        if m > s["worst"]:
            i, j = divmod(int(ratio.argmax()), ratio.shape[1])
            row = int(rows[i])
            s["worst"], s["at"] = m, (row // ITEM_ROWS, row % ITEM_ROWS, j)

    def pinned_fraction(self, name):
        s = self.out[name]
        return s["pinned"] / max(s["n"], 1)

    def ok(self):
        return all(s["bad"] == 0 for s in self.out.values())

    def failures(self):
        return {k: s for k, s in self.out.items() if s["bad"]}

    def __str__(self):
        parts = []
        for k, s in self.out.items():
            p = f" pinned {self.pinned_fraction(k):.3f}" if s["is16"] else ""
            parts.append(f"{k}: worst err/window {s['worst']:.3f} at (item, row, col) {s['at']}{p}" +
                         (f"  {s['bad']} OUT OF WINDOW, first (item, row, col, got, ref, window) {s['first_bad']}" if s["bad"] else ""))
        return "; ".join(parts)


def check_launch(ops, got, rows=None, chunk=8192, report=None):
    """check the outputs of one launch: got = {"x": X [M][D] fp32, "xn": XN 16-bit, "qkv": QKV 16-bit} (views of the first M rows,
    columns [0, D) / [0, 3D)); rows: LongTensor of the rows to check (default all)"""
    rep = report if report is not None else Report()
    M = ops.X0.shape[0]
    if rows is None:
        rows = torch.arange(M, device=ops.X0.device)
    for s in range(0, rows.numel(), chunk):
        idx = rows[s:s + chunk]
        ref = ops.rows(idx)
        for name in ("x", "xn", "qkv"):
            if name in got and got[name] is not None:
                v, w = ref[name]
                rep.add(name, idx, got[name][idx], v, w, None if name == "x" else ops.prec)
    return rep


# ------------------------------------------------------------------------------------------------------------ operand recipes
CONST_VALUES = (0.0, 1.5, -250.0)


def operands(kind, prec, D, Hd, M, seed, device="cpu", const_rows=False, large_means=False):
    """the exact operands of one launch (module docstring): 16-bit tensors in the engine's format, fp32 vectors and X rows.
    const_rows: every 7th row (from row 3) has CTX row 0 and X row = 0, 1.5 or -250, and bias_p = 0 (exact statistics);
    large_means: rows offset by 0, 20, 0, -150, 0 times their standard deviation."""
    g = torch.Generator(device=device).manual_seed(seed)
    rnd = lambda *s, sc=1.0: torch.randn(*s, generator=g, device=device) * sc
    ar = lambda n: torch.arange(n, device=device)
    q = lambda t: rn16(t.double(), prec)
    o = {"ctx": q(rnd(M, D))}
    X0 = rnd(M, D) + 0.5
    if large_means:
        offs = torch.tensor([0.0, 20.0, 0.0, -150.0, 0.0], device=device)
        X0 += offs[ar(M) % 5][:, None]
    o["g2"], o["be2"] = 1 + rnd(D, sc=0.1), rnd(D, sc=0.1)
    o["gn"], o["ben"] = 1 + rnd(D, sc=0.1), rnd(D, sc=0.1)
    o["b1"], o["b2"], o["bq"] = rnd(Hd, sc=0.2), rnd(D, sc=0.1), rnd(3 * D, sc=0.1)
    o["bp"] = rnd(D, sc=0.1)
    if kind == "dense":
        o["Wp"], o["W1"] = q(rnd(D, D, sc=0.05)), q(rnd(Hd, D, sc=0.06))
        o["W2"], o["Wq"] = q(rnd(D, Hd, sc=0.03)), q(rnd(3 * D, D, sc=0.05))
    else:
        f64 = dict(dtype=torch.float64, device=device)
        o["Wp"] = q(torch.eye(D, **f64) * 0.5)
        a = torch.tensor([0.5, -1.0, 2.0, -4.0, 1.0], **f64)
        W1 = torch.zeros(Hd, D, **f64)
        W1[ar(Hd), ar(Hd) % D] = a[ar(Hd) % 5]
        W2 = torch.zeros(D, Hd, **f64)
        W2[ar(Hd) % D, ar(Hd)] = 1.0
        Wq = torch.zeros(3 * D, D, **f64)
        Wq[ar(3 * D), ar(3 * D) % D] = torch.tensor([1.0, -0.5, 2.0], **f64)[ar(3 * D) % 3]
        o["W1"], o["W2"], o["Wq"] = q(W1), q(W2), q(Wq)
    if const_rows:
        rows = torch.arange(3, M, 7, device=device)
        o["ctx"][rows] = 0
        X0[rows] = torch.tensor(CONST_VALUES, device=device)[ar(rows.numel()) % 3][:, None]
        o["bp"] = torch.zeros(D, device=device)
    o["X0"] = X0
    return o


def fold(o, prec, fold2, foldn):
    """the folded operands vitocm_finalize_weights forms: 16-bit(W diag(gamma)), b + W beta (fp32)"""
    o = dict(o)
    if fold2:
        o["W1"], o["b1"] = rn16(o["W1"].double() * o["g2"].double(), prec), (o["b1"].double() + o["W1"].double() @ o["be2"].double()).float()
    if foldn:
        o["Wq"], o["bq"] = rn16(o["Wq"].double() * o["gn"].double(), prec), (o["bq"].double() + o["Wq"].double() @ o["ben"].double()).float()
    return o


def reference(o, prec, fold2, foldn, nxt, eps=1e-6):
    return Operands(prec, o["ctx"], o["Wp"], o["bp"], o["X0"], o["W1"], o["b1"], o["W2"], o["b2"], o["g2"], o["be2"], o["gn"], o["ben"],
                    o["Wq"], o["bq"], eps, fold2=fold2, foldn=foldn, nxt=nxt)


# ------------------------------------------------------------------------------------------------------------ unfused stages
def _acc(a, W, b):
    """a . W^T + b (float64) and its fp32 accumulation window (K + 2) 2^-24 (sum |a| |W| + |b|)"""
    a, W, b = a.double(), W.double(), b.double()
    v = a @ W.T + b
    return v, (_nnz(a, W) + 2.0) * EPS24 * (a.abs() @ W.abs().T + b.abs())


def stage_linear(a, W, b):
    """GEMM epilogue acc + bias (to 16 bits, or fp32): value and window"""
    v, w = _acc(a, W, b)
    return v, _window(v, w)


def stage_gelu(a, W, b, prec):
    """GEMM epilogue gelu(acc + bias) in the engine's sigmoid form, to 16 bits"""
    pre, wpre = _acc(a, W, b)
    h = gelu64(pre)
    return h, _window(h, GELU_ERR[prec] + GELU_APPROX_REL * pre.abs() + GELU_SLOPE * wpre)


def stage_reduce_add(X0, a, W, b):
    """GEMM epilogue X += RN(acc + bias) by the TMA reduce-add: one more rounding of the sum"""
    t, wt = _acc(a, W, b)
    x = X0.double() + t
    return x, _window(x, wt + EPS24 * x.abs())


def stage_layernorm(x, gamma, beta, eps=1e-6):
    """LayerNorm kernel (x - mean) rstd gamma + beta of exact fp32 rows, to 16 bits"""
    x = x.double()
    return _layernorm(x, torch.zeros_like(x), gamma.double(), beta.double(), eps)
