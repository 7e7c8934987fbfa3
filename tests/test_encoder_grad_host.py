"""CPU: fine-tuning the encoder -- the new kernels as ptxas builds them for sm_100a, the new C-ABI symbols, which path each state
of the gradient gate selects (on a model whose device calls are stubbed), and the refusals."""
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
from vitocm_b200.vision_transformer import _EncoderStep

CSRC = os.path.join(ROOT, "vit-ocm-wmsegmentation_b200", "csrc")

_UNIT = """
#include "train_kernels.cuh"
namespace vitocm {
void* const encoder_grad_kernels[] = {
  reinterpret_cast<void*>(grad_amax_kernel), reinterpret_cast<void*>(seed_grad_kernel<false>),
  reinterpret_cast<void*>(seed_grad_kernel<true>), reinterpret_cast<void*>(col2im_dx_kernel),
  reinterpret_cast<void*>(token_grad_kernel<false>), reinterpret_cast<void*>(token_grad_kernel<true>),
  reinterpret_cast<void*>(patch_grad_rows_kernel<false>), reinterpret_cast<void*>(patch_grad_rows_kernel<true>),
  reinterpret_cast<void*>(repack_weights_kernel),
};
}
"""


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    pytest.skip("nvcc not available")


def test_encoder_gradient_kernels_build_for_sm100a_without_spills(tmp_path):
    nvcc = _nvcc()
    src = tmp_path / "enc_grad.cu"
    src.write_text(_UNIT)
    res = subprocess.run([nvcc, "-cubin", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                          "-I", CSRC, "-o", str(tmp_path / "enc_grad.cubin"), str(src)], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    log = res.stdout + res.stderr
    spills = {name: int(st) + int(ld) for name, st, ld in
              re.findall(r"Function properties for (\S+)\n\s+\d+ bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", log)}
    for k in ("grad_amax_kernel", "seed_grad_kernel", "col2im_dx_kernel", "token_grad_kernel", "patch_grad_rows_kernel",
              "repack_weights_kernel"):
        found = [n for n in spills if k in n]
        assert found, k
        assert all(spills[n] == 0 for n in found), {n: spills[n] for n in found}


def test_new_symbols_are_exported_with_their_ctypes_signatures(lib):
    for name in ("vitocm_encoder_train_forward", "vitocm_encoder_backward"):
        assert hasattr(lib, name), name
        assert name in vob._lib.SIGNATURES
    assert len(vob._lib.SIGNATURES["vitocm_encoder_train_forward"][1]) == 11
    assert len(vob._lib.SIGNATURES["vitocm_encoder_backward"][1]) == 12
    with open(os.path.join(ROOT, "include", "vitocm.h")) as f:
        header = f.read()
    assert "int vitocm_encoder_train_forward(" in header and "int vitocm_encoder_backward(" in header


def _tiny(precision="bf16", qkv_bias=True):
    return vob.VisionTransformer(img_size=[32], patch_size=8, embed_dim=128, depth=2, num_heads=2, mlp_ratio=4, qkv_bias=qkv_bias,
                                 norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), precision=precision)


class _Spy:
    """Stubs the device calls of a model and records which path a call takes."""

    def __init__(self, m):
        self.calls = []
        feat = lambda x: torch.zeros(x.shape[0], 17, 128)   # noqa: E731
        m._encoder_train = lambda x, n: self.calls.append(("train", n)) or [feat(x)] * n
        m._forward_feats = lambda x: self.calls.append("feats") or feat(x)
        m._get_intermediate_layers = lambda x, n: self.calls.append("inter") or [feat(x)] * n


@pytest.mark.parametrize("fn", ["forward_feats", "forward", "get_intermediate_layers"])
def test_gate_selects_the_differentiable_path_only_when_asked(fn):
    m = _tiny()
    spy = _Spy(m)
    call = lambda x: getattr(m, fn)(x)   # noqa: E731
    eval_path = "inter" if fn == "get_intermediate_layers" else "feats"
    x = torch.zeros(2, 3, 32, 32)
    m.train()
    call(x)                                   # training mode, parameters require grad
    with torch.no_grad():
        call(x)                               # no_grad
        call(x.clone().requires_grad_(True))  # no_grad wins over x.requires_grad
    m.eval()
    call(x)                                   # eval(), plain x
    call(x.clone().requires_grad_(True))      # eval(), x requires grad: dx wanted
    m.train()
    m.requires_grad_(False)
    call(x)                                   # frozen encoder in training mode (linear probing)
    m.pos_embed.requires_grad_(True)
    call(x)                                   # only pos_embed trainable
    assert spy.calls == [("train", 1), eval_path, eval_path, eval_path, ("train", 1), eval_path, ("train", 1)], spy.calls


def test_fp32_parity_engines_refuse_training():
    m = _tiny("fp32").train()
    with pytest.raises(vob.VitocmError, match="bf16 or fp16"):
        m.forward_feats(torch.zeros(1, 3, 32, 32))
    with pytest.raises(vob.VitocmError, match="precision='bf16'"):
        m.get_intermediate_layers(torch.zeros(1, 3, 32, 32), n=2)


def test_gray_inputs_refuse_the_backward():
    m = _tiny().train()
    with pytest.raises(vob.VitocmError, match=r"expand\(-1, 3, -1, -1\)"):
        m.forward_feats(torch.zeros(1, 1, 32, 32))


def test_double_backward_and_overwritten_activations_are_refused():
    enc = NS(_train_ws_gen=3)
    ctx = NS(enc=enc, ws_gen=3)
    with torch.enable_grad(), pytest.raises(vob.VitocmError, match="create_graph"):
        _EncoderStep.backward(ctx, torch.zeros(1))
    ctx.ws_gen = 2
    with torch.no_grad(), pytest.raises(vob.VitocmError, match="overwritten"):
        _EncoderStep.backward(ctx, torch.zeros(1))


def test_parameters_that_get_gradients():
    """cls_token, the patch filter and bias, every block parameter and norm.* (pos_embed through dpos); no zero qkv bias."""
    m = _tiny(qkv_bias=False)
    names = set(m._encoder_grad_params())
    want = {n for n, _ in m.named_parameters()} - {"pos_embed"}
    assert names == want
    assert not any(n.endswith("attn.qkv.bias") for n in names)
    mim_enc = vob.VisionTransformerForSimMIM(patch_size=8, embed_dim=128, depth=2, num_heads=2, mlp_ratio=4, img_size=[32],
                                             qkv_bias=True, norm_layer=partial(torch.nn.LayerNorm, eps=1e-6))
    assert "mask_token" not in mim_enc._encoder_grad_params()


def test_position_graph_is_the_cached_table_and_differentiable():
    """One resize for both: the differentiable table equals the cached inference table, for square and rectangular inputs."""
    m = _tiny()
    for H, W in ((32, 32), (48, 64), (224, 224)):
        npatch = (H // 8) * (W // 8)
        g = m._pos_graph(npatch, H, W)
        assert g.requires_grad and g.shape == (npatch + 1, 128)
        ref = m._pos_graph(npatch, H, W, m.pos_embed.detach())
        assert torch.equal(g.detach(), ref)
        g.sum().backward()
        assert m.pos_embed.grad is not None
        m.pos_embed.grad = None


def test_get_intermediate_layers_with_n_below_one_returns_nothing_on_both_paths():
    m = _tiny().train()
    assert m.get_intermediate_layers(torch.zeros(1, 3, 32, 32), n=0) == []
