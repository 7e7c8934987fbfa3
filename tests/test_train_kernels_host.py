"""CPU: the kernel-level entry points of the training step's epilogues, LayerNorm backward and loss backward -- exported, declared
in the header, with ctypes signatures of the right arity -- and the LayerNorm / loss backward kernels as ptxas builds them for
sm_100a (every instantiation the step launches, no spills)."""
import os
import re
import shutil
import subprocess

import pytest

import vitocm_b200 as vob
from conftest import ROOT

CSRC = os.path.join(ROOT, "vit-ocm-wmsegmentation_b200", "csrc")

_UNIT = """
#include "train_kernels.cuh"
namespace vitocm {
void* const train_backward_kernels[] = {
  reinterpret_cast<void*>(ln_bwd_kernel<0, false>), reinterpret_cast<void*>(ln_bwd_kernel<0, true>),
  reinterpret_cast<void*>(ln_bwd_kernel<1, false>), reinterpret_cast<void*>(ln_bwd_kernel<1, true>),
  reinterpret_cast<void*>(ln_bwd_kernel<3, false>), reinterpret_cast<void*>(ln_bwd_kernel<3, true>),
  reinterpret_cast<void*>(ln_bwd_kernel<6, false>), reinterpret_cast<void*>(ln_bwd_kernel<6, true>),
  reinterpret_cast<void*>(mim_loss_bwd_kernel<false>), reinterpret_cast<void*>(mim_loss_bwd_kernel<true>),
};
}
"""

# name -> number of arguments (include/vitocm.h)
ENTRY_POINTS = {"vitocm_gemm_dgelu": 13, "vitocm_layernorm_bwd": 15, "vitocm_mim_loss_bwd": 12}


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    pytest.skip("nvcc not available")


def test_backward_kernels_build_for_sm100a_without_spills(tmp_path):
    nvcc = _nvcc()
    src = tmp_path / "train_bwd.cu"
    src.write_text(_UNIT)
    res = subprocess.run([nvcc, "-cubin", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                          "-I", CSRC, "-o", str(tmp_path / "train_bwd.cubin"), str(src)], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    log = res.stdout + res.stderr
    spills = {name: int(st) + int(ld) for name, st, ld in
              re.findall(r"Function properties for (\S+)\n\s+\d+ bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", log)}
    # mangled names: ln_bwd_kernel<NV, F16> -> ...ln_bwd_kernelILi<NV>ELb<0|1>E...
    for nv in (0, 1, 3, 6):
        for f16 in (0, 1):
            found = [n for n in spills if f"ln_bwd_kernelILi{nv}ELb{f16}E" in n]
            assert len(found) == 1, (nv, f16, sorted(spills))
            assert spills[found[0]] == 0, (found[0], spills[found[0]])
    for f16 in (0, 1):
        found = [n for n in spills if f"mim_loss_bwd_kernelILb{f16}E" in n]
        assert len(found) == 1, (f16, sorted(spills))
        assert spills[found[0]] == 0, (found[0], spills[found[0]])


def test_entry_points_are_exported_declared_and_typed(lib):
    with open(os.path.join(ROOT, "include", "vitocm.h")) as f:
        header = f.read()
    for name, arity in ENTRY_POINTS.items():
        assert hasattr(lib, name), name
        assert len(vob._lib.SIGNATURES[name][1]) == arity, name
        m = re.search(r"\bint " + name + r"\(([^;]*)\);", header)
        assert m, name
        assert len(m.group(1).split(",")) == arity, name
