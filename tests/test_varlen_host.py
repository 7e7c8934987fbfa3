"""CPU: the packing of images of different sizes (vitocm_forward_cls_attn_varlen) -- the chunk planner, the per-image offset tables
and the row -> image decode of the patch-embedding producer, the attention work items, argument refusals -- mirrored in Python, and
the new entry points present in the built library."""
import bisect

import pytest
import torch

import vitocm_b200 as vob
from vitocm_b200.vision_transformer import VARLEN_CHUNK_TOKENS, varlen_plan

SIZES = [(224, 224), (32, 32), (96, 160), (120, 136), (96, 120), (56, 56), (80, 80), (384, 384), (64, 64)]


def _attn_items(n, heads, quad_ok):
    """varlen_attn_items (vitocm_api.cu): (kernel, row0, N, query tile, first head, slots) of every work item."""
    items, row0 = [], 0
    for N in n:
        nfull, tail = divmod(N, 128)
        pack = 1 if (tail == 0 or tail > 64 or nfull > 16) else (2 if tail > 32 else 4)
        q = quad_ok and nfull >= 1
        for h in range(heads):
            for t in range(nfull):
                items.append(("quad" if q else "cta", row0, N, t, h, 1))
        if tail:
            ns = 1 if pack == 1 else (2 if q else pack)
            for h in range(0, heads, ns):
                items.append(("quad" if (q and pack > 1) else "cta", row0, N, nfull, h, ns))
        row0 += N
    return items


def test_plan_offsets_and_default_budget():
    plan = varlen_plan(SIZES, 8)
    assert plan["n"] == [(h // 8) * (w // 8) + 1 for h, w in SIZES]
    assert plan["row0"] == [sum(plan["n"][:i]) for i in range(len(SIZES))]
    assert plan["tokens"] == sum(plan["n"])
    assert plan["starts"] == [0] and plan["cap"] == plan["tokens"]   # the workspace follows the list, not the budget
    assert VARLEN_CHUNK_TOKENS == 512 * 785


def test_header_default_budget_matches():
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "include", "vitocm.h")).read()
    assert f"#define VITOCM_VARLEN_CHUNK_TOKENS {VARLEN_CHUNK_TOKENS}" in text


@pytest.mark.parametrize("budget", [1, 1000, 3000, 10 ** 9])
def test_chunk_planner(budget):
    plan = varlen_plan(SIZES, 8, budget)
    n, starts = plan["n"], plan["starts"] + [len(SIZES)]
    assert starts[0] == 0 and starts == sorted(set(starts))
    for a, b in zip(starts, starts[1:]):
        tok = sum(n[a:b])
        assert tok <= budget or b - a == 1                  # over budget only when one image alone exceeds it
        if b < len(SIZES):
            assert tok + n[b] > budget                      # closed only when the next image would not fit
        assert tok <= plan["cap"]
    if budget == 1:
        assert plan["starts"] == list(range(len(SIZES)))
    assert plan["cap"] == max(sum(n[a:b]) for a, b in zip(starts, starts[1:]))


def test_patch_row_decode():
    """GemmArgs::vimg and patch_image: every patch row maps to its image, pixel block and token row."""
    p = 8
    prefix = [0]
    for h, w in SIZES:
        prefix.append(prefix[-1] + (h // p) * (w // p))

    def patch_image(m):   # binary search of gemm_sm100.cuh
        lo, hi = 0, len(SIZES) - 1
        while lo < hi:
            mid = (lo + hi + 1) >> 1
            if prefix[mid] <= m:
                lo = mid
            else:
                hi = mid - 1
        return lo

    for m in range(prefix[-1]):
        b = patch_image(m)
        assert b == bisect.bisect_right(prefix, m) - 1
        i = m - prefix[b]
        h, w = SIZES[b]
        assert 0 <= i < (h // p) * (w // p)
        # token row = patches before + one CLS row per earlier image + this image's CLS row
        assert prefix[b] + b + 1 + i == varlen_plan(SIZES, p)["row0"][b] + 1 + i
    # image b's pixels start at C p^2 prefix[b]: the sum of the earlier images' C H W
    for b in range(len(SIZES)):
        assert 3 * p * p * prefix[b] == sum(3 * h * w for h, w in SIZES[:b])


@pytest.mark.parametrize("heads,quad_ok", [(2, True), (6, True), (3, False), (6, False)])
def test_attention_items_cover_every_query_row_once(heads, quad_ok):
    n = varlen_plan(SIZES, 8)["n"]
    items = _attn_items(n, heads, quad_ok)
    seen = {}
    for kern, row0, N, qt, h0, ns in items:
        assert ns in (1, 2, 4)
        if ns > 1:
            assert N % 128 <= 128 // ns                      # every slot holds its head's whole tail
            assert kern == "cta" or ns == 2
        slot_rows = 128 // ns
        for s in range(ns):
            h = h0 + s
            if h >= heads:
                continue                                     # computed against the last head and dropped
            for r in range(slot_rows):
                q = qt * 128 + r
                if q < N:
                    key = (row0 + q, h)
                    assert key not in seen
                    seen[key] = kern
    assert len(seen) == sum(n) * heads
    if not quad_ok:
        assert all(k == "cta" for k in seen.values())


def test_refusals_without_a_gpu():
    with pytest.raises(ValueError):
        varlen_plan([(64, 60)], 8)
    with pytest.raises(ValueError):
        varlen_plan([(0, 64)], 8)
    from functools import partial
    m = vob.VisionTransformer(img_size=[64], patch_size=8, embed_dim=128, depth=2, num_heads=2, mlp_ratio=4, qkv_bias=True,
                              norm_layer=partial(torch.nn.LayerNorm, eps=1e-6)).eval()
    with pytest.raises(ValueError):
        m.cls_attention_rows_varlen([])
    with pytest.raises(ValueError):
        m.cls_attention_rows_varlen([torch.rand(3, 64, 60)])
    with pytest.raises(ValueError):
        vob.attention_masks_varlen(m, [torch.rand(3, 64, 96)])


def test_library_exports_the_varlen_entry_points():
    lib = vob._lib.load_library()
    for s in ("vitocm_varlen_workspace_bytes", "vitocm_forward_cls_attn_varlen", "vitocm_attention_varlen", "vitocm_head_mean_varlen",
              "vitocm_tile_threshold_varlen"):
        assert hasattr(lib, s), s
        assert s in vob._lib.SIGNATURES
