"""CPU: head_dim 128 (the reference's build_model encoder: embed_dim 384, 3 heads, depth 4) through the Python mirror, and the
head_dim-128 kernels as ptxas builds them for sm_100a (no GPU needed)."""
import os
import re
import shutil
import subprocess
from types import SimpleNamespace as NS

import pytest

import vitocm_b200 as vob
from conftest import ROOT

CSRC = os.path.join(ROOT, "vit-ocm-wmsegmentation_b200", "csrc")


def test_head_dim_128_models_construct():
    m = vob.VisionTransformer(img_size=[224], patch_size=8, embed_dim=384, depth=4, num_heads=3, qkv_bias=True)
    assert m.embed_dim // m.num_heads == 128 and abs(m.qk_scale - 128 ** -0.5) < 1e-12
    args = NS(MODEL=NS(PATCH_SIZE=8), DATA=NS(IMG_SIZE=224))
    enc = vob.build_model(args, depth=4, num_heads=3)
    assert enc.depth == 4 and enc.num_heads == 3 and enc.embed_dim == 384 and len(enc.blocks) == 4
    default = vob.build_model(args)
    assert default.depth == 12 and default.num_heads == 6
    vob.VisionTransformer(img_size=[64], patch_size=8, embed_dim=256, depth=1, num_heads=2)


@pytest.mark.parametrize("embed_dim,heads", [(384, 4), (384, 12), (256, 1), (384, 5)])
def test_other_head_widths_are_refused(embed_dim, heads):
    with pytest.raises(NotImplementedError, match="64 and 128"):
        vob.VisionTransformer(img_size=[224], patch_size=8, embed_dim=embed_dim, depth=1, num_heads=heads)


_UNIT = """
#include "attention_sm100.cuh"
#include "attention_bwd_sm100.cuh"
namespace vitocm {
void* const head_dim128_kernels[] = {
#define FWD(S, P, F) reinterpret_cast<void*>(attn_fwd_tcgen05_kernel<S, 0u, P, F, 128>),
  FWD(false, false, false) FWD(false, false, true) FWD(false, true, false) FWD(false, true, true)
  FWD(true, false, false) FWD(true, false, true) FWD(true, true, false) FWD(true, true, true)
  reinterpret_cast<void*>(attn_bwd_tcgen05_kernel<128>),
};
}
"""


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    pytest.skip("nvcc not available")


def test_head_dim_128_kernels_build_for_sm100a_with_tensor_core_mmas(tmp_path):
    """Every head_dim-128 attention kernel compiles for sm_100a, issues tcgen05 MMAs (UTCHMMA in the SASS) and keeps its
    local-memory use at the level of the head_dim-64 instantiations (the setmaxnreg budgets of the kernels are per warpgroup;
    ptxas reports the register cap of the whole kernel)."""
    nvcc = _nvcc()
    src = tmp_path / "hd128.cu"
    src.write_text(_UNIT)
    cubin = tmp_path / "hd128.cubin"
    res = subprocess.run([nvcc, "-cubin", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                          "-I", CSRC, "-o", str(cubin), str(src)], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    props = dict(re.findall(r"Function properties for (\S+)\n\s+(\d+) bytes stack frame", res.stdout + res.stderr))
    kernels = [k for k in props if "Li128E" in k and ("attn_fwd_tcgen05" in k or "attn_bwd_tcgen05" in k)]
    assert len(kernels) == 9, kernels
    for k in kernels:
        assert int(props[k]) <= 256, (k, props[k])
    sass = subprocess.run([os.path.join(os.path.dirname(nvcc), "cuobjdump"), "-sass", str(cubin)], capture_output=True, text=True,
                          timeout=300).stdout
    bodies = dict(re.findall(r"Function : (\S+)\n(.*?)(?=\n\s+Function : |\Z)", sass, flags=re.S))
    for k in kernels:
        assert "UTCHMMA" in bodies[k], k
