"""GPU (B200): the attention kernels at batch sizes where every persistent CTA (every pipeline of the four-pipeline kernel) walks
several work items, so that what carries over from one item to the next -- barrier phases, the K / V and Q / dO rings, TMEM
accumulators, the O hand-over -- is exercised.  Each case:

  - asserts that the dispatch of run_attention / run_attention_bwd really gives every CTA (pipeline) of the kernel it targets at
    least two items on this device, so that a later dispatch change cannot quietly turn the case into a one-item-per-CTA test;
  - compares the kernel item by item with a float64 statement of the same op on the exact 16-bit (or hi + lo) values the kernel
    reads: forward per (image, head, 128-row query tile), dK / dV per (image, head, 128-key block[, 64-column half]), dQ per
    (image, head, query tile), each against its own reference scale, so that one wrong item among thousands cannot hide inside
    a global maximum;
  - checks that the outputs built without atomics (ctx, LSE, dK, dV) are bit-identical to those of launches over sub-batches;
  - surrounds the output with sentinel rows after row B*N and sentinel columns beyond the written width of a wider row pitch,
    which must be left untouched."""
import ctypes as C
import math

import pytest
import torch

import vitocm_b200 as vob
from gpu_util import make_engine
from vitocm_b200._lib import VitocmConfig, check, cur_stream, ptr

pytestmark = pytest.mark.gpu

BQ = 128          # query rows of a work item / keys of a backward key block (ATT_BQ)
QUAD_PIPES = 4    # pipelines per CTA of attn_fwd_quad_kernel (AQ_PIPES)
QUAD_PACK = 2     # pairs per packed tail tile in attn_fwd_quad_kernel (VITOCM_ATTN_QUAD_PACK default)
GUARD_ROWS = 64
GUARD_COLS = 64   # extra columns of the row pitch (a multiple of 8: the kernels store 16-byte vectors)
SENTINEL = {torch.bfloat16: 0x7fa5, torch.float16: 0x7e5a}   # NaN payloads no kernel produces
PREC = {"bf16": 0, "split": 1, "fp16": 2}
FWD_TOL = {"bf16": 2e-2, "fp16": 2e-3, "split": 3e-5}          # the small-shape bars of test_gpu_kernels / test_gpu_fp16
LSE_TOL = 2e-2


@pytest.fixture(autouse=True)
def _no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32 = old


def _lib():
    return vob._lib.load_library()


def _rand(shape, seed, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(shape, generator=g, device="cuda") * scale


class _Engine:
    """vitocm engine with H heads of width dh (head_dim 128 as in test_gpu_head_dim128.py), destroyed on exit."""

    def __init__(self, H, dh, precision):
        if dh == 64:
            self.h = make_engine(embed_dim=64 * H, heads=H, precision=PREC[precision])
        else:
            cfg = VitocmConfig(dh * H, 1, H, 4 * dh * H, 8, 3, 1e-6, dh ** -0.5, PREC[precision])
            self.h = C.c_void_p()
            check(_lib().vitocm_create(C.byref(cfg), C.byref(self.h)))

    def __enter__(self):
        return self.h

    def __exit__(self, *exc):
        _lib().vitocm_destroy(self.h)


# ---------------------------------------------------------------------------------------------------- dispatch: items per CTA
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def forward_plan(B, H, N, precision, dh=64, lse=False):
    """The launches of run_attention (default knobs) -> {kernel: (work items, workers)}; workers = CTAs of the generic kernel,
    pipelines (4 per CTA) of the four-pipeline kernel."""
    sms = _sms()
    tail, nfull, pairs = N % BQ, N // BQ, B * H
    pack = 1 if (tail == 0 or tail > 64 or nfull > 16) else (2 if tail > 32 else 4)
    generic = -(-pairs // pack) * (pack * nfull + (1 if tail else 0))
    plan = {}
    if dh == 64 and precision != "split" and not lse and nfull >= 1:
        tails_here = pack > 1
        quad = -(-pairs // QUAD_PACK) * (QUAD_PACK * nfull + 1) if tails_here else pairs * nfull
        plan["quad"] = (quad, min(-(-quad // QUAD_PIPES), sms) * QUAD_PIPES)
        if tail == 0 or tails_here:
            return plan
        generic = -(-pairs // pack)          # tails_only launch: one item per group's tail
    resident = sms * (1 if (precision == "split" or dh == 128) else 2)
    plan["generic"] = (generic, min(generic, resident))
    return plan


def backward_plan(B, H, N, dh=64):
    """run_attention_bwd: one item per (64-column half at head_dim 128,) key block, head, image; one CTA per SM."""
    items = -(-N // BQ) * H * B * (dh // 64)
    return {"bwd": (items, min(items, _sms()))}


def _assert_walks_items(plan, target):
    items, workers = plan[target]
    per = items // workers
    print(f"{target}: {items} items over {workers} {'pipelines' if target == 'quad' else 'CTAs'} -> >= {per} per worker "
          f"(of {_sms()} SMs)")
    assert per >= 2, f"{target}: {items} items over {workers} workers -- the case no longer walks items"
    return per


# ---------------------------------------------------------------------------------------------------- inputs, references
def _qkv(B, H, N, dh, precision, seed):
    """[B*N, 3D] activation (x 2 parts hi | lo in split mode) and rows -> the float64 values the kernel reads from those rows."""
    D = dh * H
    x = _rand((B * N, 3 * D), seed)
    if precision == "split":
        hi = x.to(torch.bfloat16)
        lo = (x - hi.float()).to(torch.bfloat16)
        qkv = torch.cat([hi, lo], 1).contiguous()
        return qkv, lambda rows: qkv[rows, :3 * D].double() + qkv[rows, 3 * D:].double()
    qkv = x.to(torch.float16 if precision == "fp16" else torch.bfloat16).contiguous()
    return qkv, lambda rows: qkv[rows].double()


def _heads(rows, B, N, H, dh):
    """[B*N, 3D] float64 -> q, k, v [B, H, N, dh]"""
    s = rows.reshape(B, N, 3, H, dh).permute(2, 0, 3, 1, 4)
    return s[0], s[1], s[2]


def _fwd_reference(exact, B, N, H, dh):
    """-> ctx [B, N, H, dh], lse2 (log2 units) [B, H, N], float64"""
    q, k, v = _heads(exact, B, N, H, dh)
    s = (q @ k.transpose(-2, -1)) * dh ** -0.5
    lse = torch.logsumexp(s, dim=-1)
    o = torch.exp(s - lse[..., None]) @ v
    return o.transpose(1, 2), lse * (1.0 / math.log(2.0))


def _tiles(x, N):
    """[b, N, ...] -> [b, ceil(N / 128), 128, ...] (zero rows pad the last tile)"""
    nq = -(-N // BQ)
    pad = torch.zeros((x.shape[0], nq * BQ - N) + tuple(x.shape[2:]), dtype=x.dtype, device=x.device)
    return torch.cat([x, pad], 1).reshape((x.shape[0], nq, BQ) + tuple(x.shape[2:]))


class _ItemErrors:
    """Per-item max |error| and max |reference| over chunks of images, and the global Frobenius sums."""

    def __init__(self, name):
        self.name, self.err, self.scale, self.num, self.den, self.images = name, [], [], 0.0, 0.0, []

    def add(self, got, ref, reduce_dims, images):
        d = (got.double() - ref)
        self.err.append(d.abs().amax(dim=reduce_dims))
        self.scale.append(ref.abs().amax(dim=reduce_dims))
        self.num += float(d.pow(2).sum())
        self.den += float(ref.pow(2).sum())
        self.images.append(images)

    def check(self, rel, absolute=0.0, global_rel=None):
        err, scale = torch.cat(self.err), torch.cat(self.scale)
        images = torch.cat(self.images)
        bar = rel * scale + absolute
        ratio = err / bar
        order = ratio.flatten().argsort(descending=True)[:4]
        worst = []
        for f in order.tolist():
            idx = list(torch.unravel_index(torch.tensor(f), ratio.shape))
            idx[0] = int(images[int(idx[0])])
            worst.append((tuple(int(i) for i in idx), f"{err.flatten()[f].item():.3e} / bar {bar.flatten()[f].item():.3e}"))
        frob = (self.num / self.den) ** 0.5
        print(f"{self.name}: {ratio.numel()} items, worst error / bar {ratio.max().item():.3f}, global relative Frobenius error "
              f"{frob:.3e}; worst items (image, ...): {worst}")
        bad = int((ratio > 1).sum())
        assert bad == 0, f"{self.name}: {bad} of {ratio.numel()} items beyond the bar; worst {worst}"
        if global_rel is not None:
            assert frob <= global_rel, (self.name, frob)


# ---------------------------------------------------------------------------------------------------- guard bands
def _guarded(rows, cols, dtype):
    """A [rows + GUARD_ROWS, cols + GUARD_COLS] buffer full of the sentinel; the kernel writes [:rows, :cols]."""
    buf = torch.empty(rows + GUARD_ROWS, cols + GUARD_COLS, device="cuda", dtype=dtype)
    buf.view(torch.int16).fill_(SENTINEL[dtype])
    return buf


def _assert_guards(buf, rows, cols, what):
    bits = buf.view(torch.int16)
    s = SENTINEL[buf.dtype]
    assert (bits[rows:] == s).all(), f"{what}: store past the last row"
    assert (bits[:rows, cols:] == s).all(), f"{what}: store beyond the written columns of the row pitch"
    assert torch.isfinite(buf[:rows, :cols].float()).all(), f"{what}: an output element was not written"


# ---------------------------------------------------------------------------------------------------- launches
def _forward(eng, qkv, B, N, D, parts, lse=None):
    """ctx in a guarded buffer (pitch D * parts + GUARD_COLS) -> the buffer"""
    out = _guarded(B * N, D * parts, qkv.dtype)
    if lse is None:
        check(_lib().vitocm_attention(eng, ptr(qkv), qkv.stride(0), B, N, ptr(out), out.stride(0), cur_stream()))
    else:
        check(_lib().vitocm_attention_fwd_lse(eng, ptr(qkv), qkv.stride(0), B, N, ptr(out), out.stride(0), ptr(lse), cur_stream()))
    torch.cuda.synchronize()
    return out


def _sub_batches(B, H, sizes):
    """[b0, b1) runs covering the batch; every run but the last holds a multiple of 4 (image, head) pairs, so that every packed
    tail tile holds the same pairs as in the launch over the whole batch"""
    out, b0, i = [], 0, 0
    while b0 < B:
        s = sizes[i % len(sizes)]
        assert (s * H) % 4 == 0
        out.append((b0, min(B, b0 + s)))
        b0 += s
        i += 1
    return out


def _sub_sizes(H, big):
    step = 4 // math.gcd(H, 4)        # images per multiple of 4 pairs
    return [step, 3 * step, big * step, 5 * step]


# ---------------------------------------------------------------------------------------------------- forward, inference
FWD_CASES = [
    # (B, H, N, dh, kernel the case walks)
    pytest.param(128, 6, 785, 64, "quad", id="quad-pack2-tails-785"),         # pack-2 tails inside the quad kernel, ~8 items / pipe
    pytest.param(128, 6, 200, 64, "generic", id="tails-only-200"),           # tail 72 > 64: quad + generic tails_only (768 / 296)
    pytest.param(16, 6, 3137, 64, "quad", id="quad-448-tile-3137"),          # > 16 full tiles: pack 1
    pytest.param(129, 3, 785, 64, "quad", id="odd-pairs-vit-tiny-785"),      # D = 192, 387 pairs: phantom pair in the last group
    pytest.param(301, 3, 150, 64, "quad", id="odd-pairs-vit-tiny-150"),
    pytest.param(32, 3, 785, 128, "generic", id="head-dim-128-785"),
]


def _check_forward(B, H, N, dh, precision, target, seed, sample=None, sub_big=8):
    plan = forward_plan(B, H, N, precision, dh)
    _assert_walks_items(plan, target)
    D, parts = dh * H, (2 if precision == "split" else 1)
    with _Engine(H, dh, precision) as eng:
        qkv, exact = _qkv(B, H, N, dh, precision, seed)
        out = _forward(eng, qkv, B, N, D, parts)
        _assert_guards(out, B * N, D * parts, "ctx")
        ctx = out[:B * N, :D * parts]
        images = torch.arange(B, device="cuda") if sample is None else sample
        errs = _ItemErrors(f"ctx {precision} {(B, H, N, dh)}")   # items: (image, query tile, head)
        chunk = max(1, (1 << 26) // (H * N * N))
        for c0 in range(0, len(images), chunk):
            idx = images[c0:c0 + chunk]
            rows = (idx[:, None] * N + torch.arange(N, device="cuda")).reshape(-1)
            ref, _ = _fwd_reference(exact(rows), len(idx), N, H, dh)
            g = (ctx[rows, :D].double() + (ctx[rows, D:].double() if parts == 2 else 0)).reshape(len(idx), N, H, dh)
            errs.add(_tiles(g, N), _tiles(ref, N), (2, 4), idx)
        errs.check(FWD_TOL[precision], global_rel=FWD_TOL[precision] / 2)
        # batch consistency: no item's result depends on the CTA / pipeline it ran on or on the items before it
        for b0, b1 in _sub_batches(B, H, _sub_sizes(H, sub_big)):
            part = _forward(eng, qkv[b0 * N:b1 * N], b1 - b0, N, D, parts)
            _assert_guards(part, (b1 - b0) * N, D * parts, "ctx (sub-batch)")
            assert torch.equal(part[:(b1 - b0) * N, :D * parts], ctx[b0 * N:b1 * N]), f"images [{b0}, {b1}) differ from the whole-batch launch"


@pytest.mark.parametrize("B,H,N,dh,target", FWD_CASES)
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_forward_16bit_many_items_per_cta(B, H, N, dh, target, precision):
    _check_forward(B, H, N, dh, precision, target, seed=100 + B + N)


@pytest.mark.parametrize("B,H,N,dh", [(64, 6, 785, 64), (32, 3, 785, 128)])
def test_forward_split_many_items_per_cta(B, H, N, dh):
    """fp32-parity mode (hi | lo operands and output): the ground truth of the masks' agreement checks."""
    _check_forward(B, H, N, dh, "split", "generic", seed=200 + B)


def test_forward_fp16_headline_batch():
    """The segmentation chunk of 2048 tiles (~80 k items of the quad kernel, ~135 per pipeline): every image bit-identical to
    launches over sub-batches, a seeded sample of 128 images item by item against float64."""
    B, H, N = 2048, 6, 785
    sample = torch.randperm(B, generator=torch.Generator().manual_seed(7))[:128].sort().values.cuda()
    _check_forward(B, H, N, 64, "fp16", "quad", seed=300, sample=sample, sub_big=128)


# ---------------------------------------------------------------------------------------------------- forward with LSE
@pytest.mark.parametrize("B,H,N,dh", [(32, 6, 785, 64), (32, 3, 785, 128)])
def test_forward_lse_many_items_per_cta(B, H, N, dh):
    """The training forward (generic kernel, LSE rows): ctx and every LSE row item by item, pad rows +inf, bit-identical to
    sub-batch launches."""
    plan = forward_plan(B, H, N, "bf16", dh, lse=True)
    _assert_walks_items(plan, "generic")
    D, npad = dh * H, -(-N // BQ) * BQ
    with _Engine(H, dh, "bf16") as eng:
        qkv, exact = _qkv(B, H, N, dh, "bf16", 400 + dh)
        lse = torch.full((B, H, npad), float("nan"), device="cuda")
        out = _forward(eng, qkv, B, N, D, 1, lse)
        _assert_guards(out, B * N, D, "ctx")
        ctx = out[:B * N, :D]
        assert torch.isinf(lse[:, :, N:]).all() and (lse[:, :, N:] > 0).all(), "pad rows of the query tiles must carry +inf"
        # items: (image, query tile, head); LSE rows against an absolute bar in log2 units
        e_ctx, e_lse = _ItemErrors(f"ctx (training forward) {(B, H, N, dh)}"), _ItemErrors(f"lse {(B, H, N, dh)}")
        for c0 in range(0, B, 8):
            c1 = min(B, c0 + 8)
            ref, ref_lse = _fwd_reference(exact(slice(c0 * N, c1 * N)), c1 - c0, N, H, dh)
            idx = torch.arange(c0, c1, device="cuda")
            e_ctx.add(_tiles(ctx[c0 * N:c1 * N].reshape(c1 - c0, N, H, dh), N), _tiles(ref, N), (2, 4), idx)
            e_lse.add(_tiles(lse[c0:c1, :, :N].transpose(1, 2), N), _tiles(ref_lse.transpose(1, 2), N), (2,), idx)
        e_ctx.check(FWD_TOL["bf16"], global_rel=FWD_TOL["bf16"] / 2)
        e_lse.check(0.0, LSE_TOL)
        for b0, b1 in _sub_batches(B, H, _sub_sizes(H, 4)):
            lp = torch.full((b1 - b0, H, npad), float("nan"), device="cuda")
            part = _forward(eng, qkv[b0 * N:b1 * N], b1 - b0, N, D, 1, lp)
            assert torch.equal(part[:(b1 - b0) * N, :D], ctx[b0 * N:b1 * N]), f"ctx of images [{b0}, {b1}) differs from the whole-batch launch"
            assert torch.equal(lp, lse[b0:b1]), f"LSE of images [{b0}, {b1}) differs from the whole-batch launch"


# ---------------------------------------------------------------------------------------------------- backward
def _bwd_reference(exact, dout, B, N, H, dh):
    """float64 dQ, dK, dV [B, N, H, dh] of ctx = softmax(scale q k^T) v"""
    q, k, v = _heads(exact, B, N, H, dh)
    do = dout.reshape(B, N, H, dh).transpose(1, 2)
    sc = dh ** -0.5
    p = torch.softmax((q @ k.transpose(-2, -1)) * sc, dim=-1)
    o = p @ v
    dv = p.transpose(-2, -1) @ do
    dp = do @ v.transpose(-2, -1)
    ds = p * (dp - (do * o).sum(-1, keepdim=True))
    dq = (ds @ k) * sc
    dk = (ds.transpose(-2, -1) @ q) * sc
    return dq.transpose(1, 2), dk.transpose(1, 2), dv.transpose(1, 2)


def _backward(eng, qkv, ctx, dctx, lse, B, N, D, H):
    """dQKV in a guarded buffer -> (buffer, dqacc after the call)"""
    npad = -(-N // BQ) * BQ
    dqkv = _guarded(B * N, 3 * D, torch.bfloat16)
    delta = torch.empty(B, H, npad, device="cuda")
    dqacc = torch.zeros(B * N, D, device="cuda")
    check(_lib().vitocm_attention_bwd(eng, ptr(qkv), qkv.stride(0), ptr(ctx), ptr(dctx), dctx.stride(0), ptr(lse), ptr(delta), ptr(dqacc),
                                      ptr(dqkv), dqkv.stride(0), B, N, cur_stream()))
    torch.cuda.synchronize()
    return dqkv, dqacc


BWD_CASES = [
    pytest.param(32, 6, 785, 64, id="mim-batch32"),          # ~9 items per CTA
    pytest.param(64, 6, 785, 64, id="mim-batch64"),
    pytest.param(40, 6, 145, 64, id="full-and-short-145"),   # one full and one 17-key block per pair
    pytest.param(40, 6, 300, 64, id="full-and-short-300"),   # 3 key blocks: with an SM count that 3 does not divide, a CTA's
                                                             # items cycle through full and short (44-key) blocks
    pytest.param(300, 2, 17, 64, id="short-blocks-17"),      # every item one short block
    pytest.param(32, 3, 785, 128, id="head-dim-128"),        # two 64-column halves per key block
]


@pytest.mark.parametrize("B,H,N,dh", BWD_CASES)
def test_backward_many_items_per_cta(B, H, N, dh):
    plan = backward_plan(B, H, N, dh)
    _assert_walks_items(plan, "bwd")
    nq, D = -(-N // BQ), dh * H
    if (B, N) == (40, 300):   # the case exists for this: block j of item it is (it / halves) % nq, items stride by the grid
        items, grid = plan["bwd"]
        js = {(it // (dh // 64)) % nq for it in range(0, items, grid)}     # the blocks CTA 0 walks
        assert js == set(range(nq)), js
    with _Engine(H, dh, "bf16") as eng:
        qkv, exact = _qkv(B, H, N, dh, "bf16", 500 + B + dh)
        dctx = (_rand((B * N, D), 501 + N, 0.5)).to(torch.bfloat16)
        npad = nq * BQ
        ctx = torch.empty(B * N, D, device="cuda", dtype=torch.bfloat16)
        lse = torch.empty(B, H, npad, device="cuda")
        check(_lib().vitocm_attention_fwd_lse(eng, ptr(qkv), qkv.stride(0), B, N, ptr(ctx), ctx.stride(0), ptr(lse), cur_stream()))
        out, dqacc = _backward(eng, qkv, ctx, dctx, lse, B, N, D, H)
        assert (dqacc == 0).all(), "dQ accumulator must be left zeroed"
        _assert_guards(out, B * N, 3 * D, "dqkv")
        dqkv = out[:B * N, :3 * D]
        halves = dh // 64
        errs = {n: _ItemErrors(f"{n} {(B, H, N, dh)}") for n in ("dq", "dk", "dv")}
        chunk = max(1, (1 << 25) // (H * N * N))
        for c0 in range(0, B, chunk):
            c1 = min(B, c0 + chunk)
            r0, r1 = c0 * N, c1 * N
            refs = _bwd_reference(exact(slice(r0, r1)), dctx[r0:r1].double(), c1 - c0, N, H, dh)
            idx = torch.arange(c0, c1, device="cuda")
            for i, (name, ref) in enumerate(zip(("dq", "dk", "dv"), refs)):
                got = dqkv[r0:r1, i * D:(i + 1) * D].reshape(c1 - c0, N, H, dh)
                if name == "dq":   # items: (image, query tile, head)
                    errs[name].add(_tiles(got, N), _tiles(ref, N), (2, 4), idx)
                else:              # items: (image, key block, head, 64-column half)
                    shape = (c1 - c0, N, H, halves, 64)
                    errs[name].add(_tiles(got.reshape(shape), N), _tiles(ref.reshape(shape), N), (2, 5), idx)
        for e in errs.values():
            e.check(3e-2, 1e-3, global_rel=1.5e-2)
        # dK / dV: one item writes each block, no atomics -> bit-identical to sub-batch launches (dQ is reduce-added in fp32
        # through L2, so its summation order varies: it is held to the item-wise bar only)
        for b0, b1 in _sub_batches(B, H, _sub_sizes(H, 4)):
            r0, r1 = b0 * N, b1 * N
            part, pacc = _backward(eng, qkv[r0:r1], ctx[r0:r1], dctx[r0:r1], lse[b0:b1], b1 - b0, N, D, H)
            assert (pacc == 0).all()
            _assert_guards(part, r1 - r0, 3 * D, "dqkv (sub-batch)")
            assert torch.equal(part[:r1 - r0, D:3 * D], dqkv[r0:r1, D:]), f"dK / dV of images [{b0}, {b1}) differ from the whole-batch launch"
