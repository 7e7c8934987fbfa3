"""CPU: the C-ABI library loads and exports every symbol include/vitocm.h declares; the Python
mirror keeps the reference's interface; host-side sharding logic (gloo, world_size 2)."""
import os
import re
import socket

import numpy as np
import pytest
import torch

import vitocm_b200 as vob
from conftest import ROOT
from oracle import vit_oracle as VO


def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "vitocm.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(vitocm_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol(lib):
    syms = _header_symbols()
    assert len(syms) >= 25
    for s in syms:
        assert hasattr(lib, s), f"libvitocm.so does not export {s}"
    assert set(syms) == set(vob._lib.SIGNATURES), "ctypes table and header disagree"
    # the block tail's two forms (plain affine, folded into the weights) take one argument list
    assert {"vitocm_block_tail", "vitocm_block_tail_folded"} <= set(syms)
    assert vob._lib.SIGNATURES["vitocm_block_tail_folded"] == vob._lib.SIGNATURES["vitocm_block_tail"]
    assert lib.vitocm_version() == 100


def test_no_compute_without_gpu_fails_loudly():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    m = vob.vit_small(patch_size=8, num_classes=0)
    with pytest.raises(vob._lib.VitocmError):
        m.get_intermediate_feat(torch.zeros(1, 3, 224, 224))
    with pytest.raises(vob._lib.VitocmError):
        vob.utils.threshold(np.zeros((8, 8), np.uint8), np.zeros((8, 8), np.float32), save=False)


def test_library_path_override_fails_loudly_when_absent(tmp_path):
    """VITOCM_LIB names another build of libvitocm.so (A/B timing of two builds on one box).  A path that does not exist must raise,
    never fall back to the in-tree library or to a CPU path; the in-tree path given explicitly loads and exports the same symbols."""
    import subprocess
    import sys
    code = ("import vitocm_b200 as v\n"
            "try:\n    v._lib.load_library(); print('LOADED', v._lib.LIB_PATH)\n"
            "except v._lib.VitocmError as e:\n    print('RAISED', e)\n")
    env = dict(os.environ, VITOCM_LIB=str(tmp_path / "no_such_libvitocm.so"))
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300).stdout
    assert out.startswith("RAISED") and "no_such_libvitocm.so" in out, out
    env["VITOCM_LIB"] = vob._lib.LIB_PATH
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300).stdout
    assert out.startswith("LOADED"), out


def test_state_dict_keys_and_param_counts_match_reference():
    m = vob.vit_small(patch_size=8, num_classes=0)
    sd_ref = VO.init_state_dict(VO.ViTConfig(**VO.VIT_SMALL))
    assert set(m.state_dict().keys()) == set(sd_ref.keys())
    for k, v in m.state_dict().items():
        assert tuple(v.shape) == tuple(sd_ref[k].shape), k
    assert sum(p.numel() for p in m.parameters()) == 21670272          # SSS/output/log_rank0.txt:5570
    m.load_state_dict(sd_ref, strict=True)
    b = vob.vit_base(patch_size=8, num_classes=0)
    assert b.embed_dim == 768 and b.num_heads == 12 and b.patch_embed.patch_size == 8
    assert m.num_features == 384 and len(m.blocks) == 12


def test_init_distributions_follow_reference():
    torch.manual_seed(0)
    m = vob.vit_small(patch_size=8, num_classes=0)
    w = m.blocks[3].mlp.fc1.weight
    assert abs(w.std().item() - 0.02) < 1e-3 and w.abs().max().item() <= 2.0
    assert torch.all(m.blocks[0].attn.qkv.bias == 0) and torch.all(m.norm.weight == 1)
    assert m.norm.eps == 1e-6


def test_lazy_attention_serves_cls_row_without_materialising():
    rows = torch.arange(2 * 3 * 5, dtype=torch.float32).reshape(2, 3, 5)
    calls = []

    def producer():
        calls.append(1)
        full = torch.zeros(2, 3, 5, 5)
        full[:, :, 0, :] = rows
        return full

    la = vob.LazyAttention((2, 3, 5, 5), producer, rows)
    got = la[0, :, 0, 1:]
    assert torch.equal(got, rows[0, :, 1:]) and not calls
    assert la.shape == (2, 3, 5, 5) and la.shape[1] == 3
    assert torch.equal(la[1, :, 0, :], rows[1])
    _ = la[0, :, 2, 1:]
    assert calls == [1]
    assert torch.equal(torch.as_tensor(la.materialize())[:, :, 0], rows)


def test_shard_range_and_grid_size():
    for total in (1, 7, 145, 1225, 21025):
        for world in (1, 2, 3, 8):
            spans = [vob.shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1
    assert vob.grid_size(4096, 112) == 35 and vob.grid_size(16384, 112) == 145 and vob.grid_size(1152, 128) == 7


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_worker(rank, world, port, tmp):
    import torch.distributed as dist
    import vitocm_b200 as v
    from vitocm_b200 import sw_processing as sw
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        T, E = 25, 37
        g = torch.Generator().manual_seed(0)
        maps = torch.rand(T, 4, 4, generator=g)
        a, b = v.shard_range(T, rank, world)
        full = sw.allgather_shards(maps[a:b].clone(), T, rank, world)
        assert torch.equal(full, maps)
        mask = (torch.rand(E, 9, generator=g) > 0.5).to(torch.uint8)
        y0, y1 = v.shard_range(E, rank, world)
        got = sw.gather_bands(mask[y0:y1].clone(), E, rank, world, dst=0)
        if rank == 0:
            assert torch.equal(got, mask)
        else:
            assert got is None
        # two results of the same shape gathered back to back stay distinct (one receive buffer per tag) -- bands that divide
        # evenly come back as the receive buffer itself
        E2 = 36
        m1 = (torch.rand(E2, 9, generator=g) > 0.5).to(torch.uint8)
        m2 = 1 - m1
        z0, z1 = v.shard_range(E2, rank, world)
        g1 = sw.gather_bands(m1[z0:z1].clone(), E2, rank, world, dst=0, tag="th")
        g2 = sw.gather_bands(m2[z0:z1].clone(), E2, rank, world, dst=0, tag="th3")
        if rank == 0:
            assert torch.equal(g1, m1) and torch.equal(g2, m2)
        mm = torch.tensor([100 + rank, 7 - rank], dtype=torch.int32)
        sw.allreduce_minmax(mm)
        assert mm.tolist() == [100, 7]
        hist = torch.full((3, 256), rank + 1, dtype=torch.int64)
        dist.all_reduce(hist)
        assert int(hist[0, 0]) == sum(range(1, world + 1))
        # MIM data parallelism: the flat gradient buffer is summed over ranks (DataParallel + loss.sum(), SSS/mim.py:102,174)
        from functools import partial
        enc = v.VisionTransformerForSimMIM(patch_size=8, embed_dim=128, depth=1, num_heads=2, mlp_ratio=4, img_size=[32], qkv_bias=True,
                                           norm_layer=partial(torch.nn.LayerNorm, eps=1e-6))
        mim = v.MIM(encoder=enc, encoder_stride=8)
        mim._gflat = torch.arange(10, dtype=torch.float32) * (rank + 1)
        mim.all_reduce_grads()
        assert torch.equal(mim._gflat, torch.arange(10, dtype=torch.float32) * sum(range(1, world + 1)))
        open(os.path.join(tmp, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_multi_rank_host_logic_gloo_world2(tmp_path):
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_gloo_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


def test_checkpoint_file_round_trip_on_the_host(tmp_path):
    """SURVEY.md 8(f) rank 4 (host half; no compute): save_checkpoint writes the reference's dictionary
    (SSS/utils.py:375-385) and load_pretrained_weights applies eval.py:67-77's key handling."""
    from functools import partial
    from types import SimpleNamespace as NS
    import torch
    import vitocm_b200 as vob

    torch.manual_seed(3)
    mk = lambda: vob.VisionTransformer(patch_size=8, embed_dim=64, depth=1, num_heads=1, mlp_ratio=4, img_size=[16], qkv_bias=True,
                                       norm_layer=partial(torch.nn.LayerNorm, eps=1e-6))
    a, b = mk(), mk()
    opt = torch.optim.AdamW(a.parameters(), lr=1e-3)
    sched = vob.lr_scheduler.CosineLRScheduler(opt, t_initial=10, lr_min=1e-6, warmup_t=0, warmup_lr_init=0.0)
    path = vob.utils.save_checkpoint(NS(OUTPUT=str(tmp_path)), 7, a, 0.5, opt, sched, None)
    assert path.endswith("ckpt_epoch_7.pth")
    msg = vob.utils.load_pretrained_weights(b, path)
    assert msg.missing_keys == [] and msg.unexpected_keys == []
    assert all(torch.equal(v, b.state_dict()[k]) for k, v in a.state_dict().items())
    # DataParallel / multicrop-wrapper prefixes on the top-level keys and a checkpoint_key, as eval.py handles them
    ck = torch.load(path, map_location="cpu", weights_only=False)
    torch.save({"teacher": {"module.model": ck["model"]}}, tmp_path / "wrapped.pth")
    c = mk()
    vob.utils.load_pretrained_weights(c, str(tmp_path / "wrapped.pth"), checkpoint_key="teacher")
    assert all(torch.equal(v, c.state_dict()[k]) for k, v in a.state_dict().items())
