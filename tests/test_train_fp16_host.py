"""CPU: fp16 training -- the fp16 instantiations of the weight-gradient GEMM and the attention backward as ptxas builds them for
sm_100a (no GPU needed), and fp16 MIM encoders through the Python mirror."""
import os
import re
import shutil
import subprocess
from types import SimpleNamespace as NS

import pytest

import vitocm_b200 as vob
from conftest import ROOT

CSRC = os.path.join(ROOT, "vit-ocm-wmsegmentation_b200", "csrc")

_UNIT = """
#include "wgrad_sm100.cuh"
#include "attention_bwd_sm100.cuh"
namespace vitocm {
void* const train_kernels[] = {
#define WG(BN, NB) reinterpret_cast<void*>(wgrad_bf16_tcgen05_kernel<BN, NB, false>), reinterpret_cast<void*>(wgrad_bf16_tcgen05_kernel<BN, NB, true>),
  WG(64, 1) WG(128, 1) WG(192, 1) WG(256, 1) WG(192, 2)
  reinterpret_cast<void*>(attn_bwd_tcgen05_kernel<64, false>), reinterpret_cast<void*>(attn_bwd_tcgen05_kernel<64, true>),
  reinterpret_cast<void*>(attn_bwd_tcgen05_kernel<128, false>), reinterpret_cast<void*>(attn_bwd_tcgen05_kernel<128, true>),
};
}
"""


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    pytest.skip("nvcc not available")


def test_fp16_training_kernels_build_for_sm100a_with_tensor_core_mmas(tmp_path):
    """Every fp16 weight-gradient and attention-backward instantiation compiles for sm_100a, issues tcgen05 MMAs (UTCHMMA) and
    spills no more than its bf16 twin."""
    nvcc = _nvcc()
    src = tmp_path / "train16.cu"
    src.write_text(_UNIT)
    cubin = tmp_path / "train16.cubin"
    res = subprocess.run([nvcc, "-cubin", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                          "-I", CSRC, "-o", str(cubin), str(src)], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    log = res.stdout + res.stderr
    spills = {name: int(st) + int(ld) for name, st, ld in
              re.findall(r"Function properties for (\S+)\n\s+\d+ bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", log)}
    kernels = [k for k in spills if "wgrad_bf16_tcgen05" in k or "attn_bwd_tcgen05" in k]
    assert len(kernels) == 14, kernels
    sass = subprocess.run([os.path.join(os.path.dirname(nvcc), "cuobjdump"), "-sass", str(cubin)], capture_output=True, text=True,
                          timeout=300).stdout
    bodies = dict(re.findall(r"Function : (\S+)\n(.*?)(?=\n\s+Function : |\Z)", sass, flags=re.S))
    f16 = [k for k in kernels if "ELb1EEEv" in k]
    assert len(f16) == 7, f16
    for k in f16:
        twin = k.replace("ELb1EEEv", "ELb0EEEv")
        assert twin in spills, twin
        assert "UTCHMMA" in bodies[k], k
        assert spills[k] <= spills[twin], (k, spills[k], spills[twin])


def test_fp16_mim_encoders_construct():
    enc = vob.VisionTransformerForSimMIM(patch_size=8, embed_dim=384, depth=4, num_heads=3, img_size=[224], qkv_bias=True, precision="fp16")
    assert enc.precision == "fp16"
    mim = vob.MIM(encoder=enc, encoder_stride=8)
    assert mim.encoder is enc
    args = NS(MODEL=NS(PATCH_SIZE=8), DATA=NS(IMG_SIZE=224))
    built = vob.build_model(args, depth=4, num_heads=3, precision="fp16")
    assert built.precision == "fp16" and built.depth == 4 and built.num_heads == 3
    assert vob.build_model(args).precision == "bf16"          # the default training precision is unchanged
