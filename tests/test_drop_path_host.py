"""CPU: stochastic depth (drop_path_rate) -- the rate checks and DINO's schedule, the scale draws against a restatement of the
reference's drop_path calls, the new C-ABI symbols, the scaled GEMM / LayerNorm-backward instantiations as ptxas builds them for
sm_100a, and which path each model state selects (device calls stubbed), including the training-mode refusals."""
import os
import re
import shutil
import subprocess
from functools import partial
from types import SimpleNamespace as NS

import pytest
import torch

import vitocm_b200 as vob
from conftest import ROOT
from vitocm_b200.vision_transformer import draw_branch_scales

CSRC = os.path.join(ROOT, "vit-ocm-wmsegmentation_b200", "csrc")


def _tiny(rate=0.0, precision="bf16", depth=4):
    return vob.VisionTransformer(img_size=[32], patch_size=8, embed_dim=128, depth=depth, num_heads=2, mlp_ratio=4, qkv_bias=True,
                                 norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), precision=precision, drop_path_rate=rate)


# ------------------------------------------------------------------------------------------------------------ constructor
@pytest.mark.parametrize("rate", [-0.1, 1.0, 1.5, float("nan")])
def test_rates_outside_zero_one_are_refused(rate):
    with pytest.raises(ValueError, match="drop_path_rate"):
        _tiny(rate)


def test_dropout_rates_stay_refused():
    with pytest.raises(NotImplementedError):
        vob.VisionTransformer(img_size=[32], patch_size=8, embed_dim=128, depth=2, num_heads=2, drop_rate=0.1)
    with pytest.raises(NotImplementedError):
        vob.VisionTransformer(img_size=[32], patch_size=8, embed_dim=128, depth=2, num_heads=2, attn_drop_rate=0.1)


@pytest.mark.parametrize("rate,depth", [(0.1, 12), (0.3, 4), (0.0, 3), (0.5, 1)])
def test_schedule_is_dinos_and_parameter_free(rate, depth):
    m = _tiny(rate, depth=depth)
    want = [v.item() for v in torch.linspace(0, rate, depth)]      # vit.py:155
    assert [b.drop_path.drop_prob for b in m.blocks] == want
    assert m.blocks[0].drop_path.drop_prob == 0.0
    assert set(m.state_dict()) == set(_tiny(0.0, depth=depth).state_dict())
    assert not list(m.blocks[0].drop_path.parameters())


def test_dinos_vit_small_arguments_construct():
    m = vob.vit_small(patch_size=8, drop_path_rate=0.1)               # DINO's student
    assert m.blocks[-1].drop_path.drop_prob == pytest.approx(0.1)


def test_build_model_takes_drop_path_rate():
    args = NS(MODEL=NS(PATCH_SIZE=8), DATA=NS(IMG_SIZE=192))
    assert all(b.drop_path.drop_prob == 0.0 for b in vob.model.build_model(args, depth=4, num_heads=3).blocks)
    enc = vob.model.build_model(args, depth=4, num_heads=3, drop_path_rate=0.1)
    assert enc.blocks[-1].drop_path.drop_prob == pytest.approx(0.1)


# ------------------------------------------------------------------------------------------------------------ the draws
def _reference_drop_path(x, drop_prob, training):
    """SSS/dino/vision_transformer.py drop_path, verbatim in substance"""
    if drop_prob == 0. or not training:
        return x
    keep_prob = 1 - drop_prob
    shape = (x.shape[0],) + (1,) * (x.ndim - 1)
    random_tensor = keep_prob + torch.rand(shape, dtype=x.dtype, device=x.device)
    random_tensor.floor_()
    return x.div(keep_prob) * random_tensor


def _reference_scales(probs, B, seed):
    """The reference's Block.forward calls in order (attn branch, then mlp branch, block by block; nn.Identity for rate 0) on
    branch outputs of ones: what each sample's branch is multiplied by."""
    torch.manual_seed(seed)
    out = torch.ones(len(probs), 2, B)
    for l, p in enumerate(probs):
        for k in range(2):
            if p > 0:
                out[l, k] = _reference_drop_path(torch.ones(B, 1, 1), p, True).reshape(B)
    return out


@pytest.mark.parametrize("rate,depth,B", [(0.1, 12, 32), (0.5, 4, 64), (0.9, 3, 7)])
def test_draws_match_the_reference_calls_in_order(rate, depth, B):
    probs = [v.item() for v in torch.linspace(0, rate, depth)]
    ref = _reference_scales(probs, B, seed=1234)
    torch.manual_seed(1234)
    got = draw_branch_scales(probs, B, "cpu")
    assert got.shape == (depth, 2, B) and got.dtype == torch.float32
    assert torch.equal(got, ref)
    # the same number of draws: the generators end in the same state
    after = torch.rand(4)
    _reference_scales(probs, B, seed=1234)
    assert torch.equal(torch.rand(4), after)
    assert torch.equal(got[0], torch.ones(2, B))                    # block 0 never drops and draws nothing


def test_rate_zero_draws_nothing():
    torch.manual_seed(5)
    s = draw_branch_scales([0.0, 0.0], 3, "cpu")
    assert torch.equal(s, torch.ones(2, 2, 3))
    after = torch.rand(1)
    torch.manual_seed(5)
    assert torch.equal(torch.rand(1), after)


# ------------------------------------------------------------------------------------------------------------ C ABI
# name -> number of arguments (include/vitocm.h)
ENTRY_POINTS = {"vitocm_mim_train_forward_dp": 13, "vitocm_encoder_train_forward_dp": 12, "vitocm_gemm_resid_scaled": 14,
                "vitocm_layernorm_bwd_scaled": 17}


def test_new_symbols_are_exported_declared_and_typed(lib):
    with open(os.path.join(ROOT, "include", "vitocm.h")) as f:
        header = f.read()
    for name, arity in ENTRY_POINTS.items():
        assert hasattr(lib, name), name
        assert len(vob._lib.SIGNATURES[name][1]) == arity, name
        m = re.search(r"\bint " + name + r"\(([^;]*)\);", header)
        assert m, name
        assert len(m.group(1).split(",")) == arity, name
    assert lib.vitocm_version() == 100


_UNIT = """
#include "train_kernels.cuh"
namespace vitocm {
void* const drop_path_kernels[] = {
  reinterpret_cast<void*>(ln_bwd_kernel<0, false, true>), reinterpret_cast<void*>(ln_bwd_kernel<0, true, true>),
  reinterpret_cast<void*>(ln_bwd_kernel<1, false, true>), reinterpret_cast<void*>(ln_bwd_kernel<1, true, true>),
  reinterpret_cast<void*>(ln_bwd_kernel<3, false, true>), reinterpret_cast<void*>(ln_bwd_kernel<3, true, true>),
  reinterpret_cast<void*>(ln_bwd_kernel<6, false, true>), reinterpret_cast<void*>(ln_bwd_kernel<6, true, true>),
  reinterpret_cast<void*>(gemm_bf16_tcgen05_kernel<64, EPI_RESID_SCALED_F32, false>),
  reinterpret_cast<void*>(gemm_bf16_tcgen05_kernel<128, EPI_RESID_SCALED_F32, false>),
  reinterpret_cast<void*>(gemm_bf16_tcgen05_kernel<192, EPI_RESID_SCALED_F32, false>),
  reinterpret_cast<void*>(gemm_bf16_tcgen05_kernel<256, EPI_RESID_SCALED_F32, false>),
  reinterpret_cast<void*>(gemm_bf16_tcgen05_kernel<128, EPI_RESID_SCALED_F32, false, true>),
  reinterpret_cast<void*>(gemm_bf16_tcgen05_kernel<192, EPI_RESID_SCALED_F32, false, true>),
  reinterpret_cast<void*>(gemm_bf16_tcgen05_kernel<128, EPI_RESID_SCALED_F32, false, false, 1, true>),
  reinterpret_cast<void*>(gemm_bf16_tcgen05_kernel<192, EPI_RESID_SCALED_F32, false, false, 1, true>),
  reinterpret_cast<void*>(gemm_bf16_tcgen05_kernel<256, EPI_RESID_SCALED_F32, false, false, 1, true>),
};
}
"""


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    pytest.skip("nvcc not available")


def test_scaled_instantiations_build_for_sm100a_without_spills(tmp_path):
    """The scaled residual epilogue (single CTA at every tile width, B-resident at 128 / 192, CTA pairs at 128 / 192 / 256) and the
    scaled LayerNorm backward for every NV, bf16 and fp16."""
    src = tmp_path / "drop_path.cu"
    src.write_text(_UNIT)
    res = subprocess.run([_nvcc(), "-cubin", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                          "-I", CSRC, "-o", str(tmp_path / "drop_path.cubin"), str(src)], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    log = res.stdout + res.stderr
    spills = {name: int(st) + int(ld) for name, st, ld in
              re.findall(r"Function properties for (\S+)\n\s+\d+ bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", log)}
    # mangled: ln_bwd_kernel<NV, F16, true> -> ...ln_bwd_kernelILi<NV>ELb<F16>ELb1EE..., the GEMM's EPI = 7 -> ...kernelILi<BN>ELi7E...
    ln = [n for n in spills if re.search(r"ln_bwd_kernelILi\dELb[01]ELb1EE", n)]
    gemm = [n for n in spills if re.search(r"gemm_bf16_tcgen05_kernelILi\d+ELi7E", n)]
    assert len(ln) == 8, sorted(spills)
    assert len(gemm) == 9, sorted(spills)
    assert all(spills[n] == 0 for n in ln + gemm), {n: spills[n] for n in ln + gemm if spills[n]}


# ------------------------------------------------------------------------------------------------------------ path selection
class _Spy:
    """Stubs the device calls of a model and records which path a call takes."""

    def __init__(self, m):
        self.calls = []
        feat = lambda x: torch.zeros(x.shape[0], 17, 128)   # noqa: E731
        m._encoder_train = lambda x, n: self.calls.append(("train", n)) or [feat(x)] * n
        m._forward_feats = lambda x: self.calls.append("feats") or feat(x)
        m._get_intermediate_layers = lambda x, n: self.calls.append("inter") or [feat(x)] * n


@pytest.mark.parametrize("fn", ["forward_feats", "forward", "get_intermediate_layers"])
def test_train_mode_drops_paths_under_no_grad_too(fn):
    x = torch.zeros(2, 3, 32, 32)
    eval_path = "inter" if fn == "get_intermediate_layers" else "feats"
    for rate, want_no_grad in ((0.2, ("train", 1)), (0.0, eval_path)):
        m = _tiny(rate)
        spy = _Spy(m)
        call = lambda: getattr(m, fn)(x)   # noqa: E731
        m.train()
        call()                                  # training mode, gradients: the training forward either way
        with torch.no_grad():
            call()                              # no_grad: the reference still drops paths in training mode
        m.requires_grad_(False)
        call()                                  # frozen model in training mode: still dropped when the rate is positive
        m.eval()
        call()                                  # eval(): inference path, drop path is the identity
        with torch.no_grad():
            call()
        assert spy.calls == [("train", 1), want_no_grad, want_no_grad, eval_path, eval_path], (rate, spy.calls)


def test_branch_scales_only_in_training_mode_with_a_positive_rate():
    m = _tiny(0.3, depth=3)
    assert m.train()._branch_scales(5, "cpu").shape == (3, 2, 5)
    assert m.eval()._branch_scales(5, "cpu") is None
    assert _tiny(0.0).train()._branch_scales(5, "cpu") is None


@pytest.mark.parametrize("call", [
    lambda m, x: m.cls_attention_rows(x),
    lambda m, x: m.get_last_selfattention(x),
    lambda m, x: m.get_intermediate_feat(x),
    lambda m, x: m.get_intermediate_feat(x, n=2, lazy=False),
    lambda m, x: m.attention_rows(x, [0]),
    lambda m, x: m.cls_attention_rows_mosaic(torch.zeros(64, 64, dtype=torch.uint8), 2, 32, 32, 0, 4),
], ids=["cls_attention_rows", "get_last_selfattention", "get_intermediate_feat", "get_intermediate_feat_full", "attention_rows",
        "mosaic"])
def test_attention_maps_refuse_training_mode_with_drop_path(call):
    m = _tiny(0.1).train()
    with pytest.raises(vob.VitocmError, match=r"\.eval\(\)"):
        call(m, torch.zeros(1, 3, 32, 32))


def test_simmim_encoder_forward_refuses_training_mode_with_drop_path():
    enc = vob.VisionTransformerForSimMIM(patch_size=8, embed_dim=128, depth=2, num_heads=2, mlp_ratio=4, img_size=[32], qkv_bias=True,
                                         norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), drop_path_rate=0.1).train()
    with pytest.raises(vob.VitocmError, match=r"\.eval\(\)"):
        enc(torch.zeros(1, 3, 32, 32), torch.zeros(1, 4, 4))


@pytest.mark.parametrize("rate", [0.0, 0.2])
def test_mim_forward_path_selection(rate):
    enc = vob.VisionTransformerForSimMIM(patch_size=8, embed_dim=128, depth=2, num_heads=2, mlp_ratio=4, img_size=[32], qkv_bias=True,
                                         norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), drop_path_rate=rate)
    mim = vob.MIM(encoder=enc, encoder_stride=8)
    calls = []
    mim._forward_train = lambda x, m: calls.append(("train", torch.is_grad_enabled())) or (None, None, None)
    mim._forward_eval = lambda x, m: calls.append("eval") or (None, None, None)
    x, mask = torch.zeros(1, 3, 32, 32), torch.zeros(1, 4, 4)
    mim.train()
    mim(x, mask)
    with torch.no_grad():
        mim(x, mask)
    mim.eval()
    mim(x, mask)
    dropped = ("train", False) if rate > 0 else "eval"
    assert calls == [("train", True), dropped, "eval"], calls


def test_fp32_parity_engines_refuse_drop_path_in_training_mode():
    m = _tiny(0.1, precision="fp32").train()
    with torch.no_grad(), pytest.raises(vob.VitocmError, match=r"\.eval\(\)"):
        m.forward_feats(torch.zeros(1, 3, 32, 32))
