#!/usr/bin/env python
"""bench.py -- sliding-window segmentation throughput of the ViT-OCM hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
    python bench.py --impl reference --steps K --warmup W    (CPU arm: the reference algorithm on host cores)
    python bench.py ... --dump-outputs DIR                   (also write the outputs of the last timed step: dump_outputs)

One "step" = one pass of the whole hot path over one synthetic gray mosaic: sliding window ->
ViT-S/8 CLS attention rows per 224x224 tile -> head mean / per-tile min-max / bilinear / ramp-blended
stitch -> global min-max -> img*att -> Otsu -> masks.  N=1 is BASELINE.json configs[1] (4096x4096,
window 224, stride 112 -> 35x35 = 1225 tiles, stitched extent 4032^2 = 16.257 MP).  For N>1 the
mosaic grows so that tiles per GPU stay ~1225 (weak scaling); tiles shard over ranks, low-res maps are
all-gathered, {min,max,histograms} all-reduced and the mask bands gathered on rank 0.
Prints ONE JSON line on rank 0.

Precision: the headline runs fp16 engines (IEEE half tensor-core operands, fp32 accumulate / residual / LN / softmax statistics):
same tensor-core rate as bf16 and 8x less operand rounding -- the reference is an fp32 model and its masks only agree on >= 99.9 %
of the pixels when the CLS rows are good to ~1e-4 (DESIGN.md section 4).  The line carries `mask_agreement` (this run's masks
against the fp32-parity mode on the same mosaic), `precision_modes` (throughput + agreement of bf16 / fp16+mlp2 / fp32 on the
same box), `cfg3` (BASELINE configs[2]: ViT-B/8, fixed 16384^2 mosaic, strong scaling), `mim_train` (configs[3], batch 32 per
GPU) and, for N > 1, `multi_gpu_bitwise_equal` (rank 0 re-segments the whole mosaic alone and compares the bits).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WINDOW, STRIDE, PATCH = 224, 112, 8
ARCHS = {"vit_small": dict(embed_dim=384, depth=12, num_heads=6), "vit_base": dict(embed_dim=768, depth=12, num_heads=12)}
METRIC = "sliding_window_seg_megapixels_per_s"


def flops_per_tile(D, depth, heads, N):
    """Algorithmic FLOPs of the CLS-row path per tile (BASELINE.md section 4): patch-embed, depth-1 full
    blocks, last block K projection + q_cls.K^T; 2*M*N*K per contraction, softmax/LN/GELU excluded."""
    n = N - 1
    pe = 2 * n * (3 * PATCH * PATCH) * D
    blk = 2 * N * D * 3 * D + 4 * N * N * D + 2 * N * D * D + 16 * N * D * D
    last = 2 * N * D * D + 2 * D * D + 2 * N * D
    return pe + (depth - 1) * blk + last


def class_flops(cls, D, N, tiles, depth):
    """Algorithmic FLOPs of all launches of one kernel class in a step."""
    M = tiles * N
    L = depth - 1
    return {"gemm_qkv": 2 * M * D * 3 * D * L, "gemm_proj": 2 * M * D * D * L, "gemm_fc1_gelu": 2 * M * D * 4 * D * L,
            "gemm_fc2": 2 * M * 4 * D * D * L, "mlp_fused": 4 * M * 4 * D * D * L, "block_tail": (2 * M * D * D + 4 * M * 4 * D * D) * L, "attention": 4 * tiles * N * N * D * L, "gemm_k_last": 2 * M * D * D,
            "patch_embed": 2 * tiles * (N - 1) * 192 * D}.get(cls, 0)


def mosaic_geometry(n_gpus):
    n = int(round(35 * math.sqrt(n_gpus)))
    size = (n + 1) * STRIDE + 64          # range(0, size - 2*STRIDE, STRIDE) has exactly n origins; 4096 for n = 35
    extent = (n - 1) * STRIDE + WINDOW
    return n, size, extent


class ClockSampler(threading.Thread):
    """Clocks / throttle reasons of one GPU while the timed region runs (the recipe's clocks line).  Sampled IN PROCESS through NVML
    (nvidia_ml_py: SM clock, max SM clock, clocks-event reasons every 150 ms) -- a long-lived `nvidia-smi -lms 200` next to the bench
    cost single timed steps 50-450 ms now and then (profiles/r02_gpu_call_al_final.log, r02_gpu_call_am_bench_spread.log: its
    queries include power.draw and run through a second process); `nvidia-smi` remains the fall-back when NVML cannot be loaded.
    `open_window()` / `stop()` bracket the timed region and only samples taken inside it count.  Only the rank that prints the JSON
    line samples (enabled=False elsewhere)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index, enabled=True):
        super().__init__(daemon=True)
        self.index, self.enabled = index, enabled
        self.raw, self.samples, self.t_open, self.t_close, self.proc = [], [], None, None, None
        self.nvml, self.handle, self.halt = None, None, threading.Event()
        if not enabled:
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            try:   # the CUDA device's own NVML handle (CUDA_VISIBLE_DEVICES may renumber)
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml
        except Exception:
            self.nvml = None
            try:
                self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                              "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            except Exception:
                self.proc = None

    def run(self):
        if self.nvml is not None:
            nv = self.nvml
            reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self.halt.is_set():
                try:
                    sm = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                    bits = int(reasons_fn(self.handle))
                    self.raw.append((time.perf_counter(), [str(sm), str(self.max_sm), ""] +
                                     ["Active" if bits & mask else "Not Active" for _, mask in self.BITS]))
                except Exception:
                    pass
                self.halt.wait(0.15)
            return
        if self.proc is None:
            return
        for line in self.proc.stdout:
            line = line.strip()
            if line:
                self.raw.append((time.perf_counter(), [s.strip() for s in line.split(",")]))

    def open_window(self):
        self.t_open = time.perf_counter()

    def stop(self):
        self.t_close = time.perf_counter()
        self.halt.set()
        if self.proc is not None:
            try:
                self.proc.terminate()
                self.proc.wait(timeout=3)
            except Exception:
                pass
        self.join(timeout=3)
        inside = [v for t, v in self.raw if self.t_open is not None and self.t_open <= t <= self.t_close]
        self.samples = inside if inside else [v for _, v in self.raw[-2:]]   # a region shorter than one sampling period

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples if len(s) >= 7 for i in range(4) if s[3 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------- CPU arm
def cpu_reference_sample(arch, threads, n_s=3, repeats=1):
    """The reference algorithm (oracle port, torch-CPU fp32 + numpy) on a bounded sample: n_s x n_s tiles
    through get_intermediate_feat -> compute_attention -> mean -> per-tile min-max -> resize pair, then
    concat_crops + threshold.  Returns (tiles_per_s, post_s_per_MP, sample description)."""
    from oracle import post_oracle as PO
    from oracle import vit_oracle as VO
    torch.set_num_threads(threads)
    cfg = VO.ViTConfig(**ARCHS[arch])
    sd = VO.init_state_dict(cfg, seed=0)
    size = (n_s + 1) * STRIDE + 64
    mosaic = VO.synthetic_mosaic_u8(size, seed=4321)
    crops = PO.sliding_window(mosaic, STRIDE, WINDOW)
    t_tiles = t_post = 0.0
    for _ in range(repeats):
        t0 = time.perf_counter()
        rows = []
        for c in crops:                                           # serial, batch 1, like the reference loop
            x = torch.from_numpy(c).float().div(255.0)[None, None].expand(1, 3, -1, -1).contiguous()
            feat, attns, qkvs = VO.get_intermediate_feat(sd, cfg, x, n=1)
            rows.append(attns[0][0, :, 0, :].numpy())
        t1 = time.perf_counter()
        stitched, masks, gray = PO.mosaic_segment(np.stack(rows), mosaic, STRIDE, WINDOW, PATCH)
        t2 = time.perf_counter()
        t_tiles += t1 - t0
        t_post += t2 - t1
    ntiles = len(crops) * repeats
    ext = (n_s - 1) * STRIDE + WINDOW
    return ntiles / t_tiles, t_post / (repeats * ext * ext / 1e6), f"{n_s}x{n_s} tiles of {arch}/8 ({WINDOW}^2, stride {STRIDE}) + stitch/threshold of the {ext}^2 extent, x{repeats}"


def cpu_value(tiles_per_s, post_s_per_mp, n_tiles, extent):
    mp = extent * extent / 1e6
    return mp / (n_tiles / tiles_per_s + post_s_per_mp * mp)



def workload_config(arch, n_gpus, precision="fp16", chunk_tiles=2048, lanes=1):
    """config dict of the segmentation workload at n_gpus ranks -- the SAME keys and strings in the GPU arm and the reference arm."""
    n, size, extent = mosaic_geometry(n_gpus)
    T = n * n
    return {"workload": f"{arch}/8 sliding-window segmentation, {size}x{size} gray mosaic, window {WINDOW}, stride {STRIDE}, "
                        f"{T} tiles, extent {extent}^2", "tiles": T, "tiles_per_gpu": -(-T // n_gpus), "weights": "random init (seed 0)",
            "chunk_tiles": chunk_tiles, "lanes": lanes, "precision": precision,
            "l2": "flushed between timed steps (256 MiB write, untimed); per-step working set >> L2",
            "parallelism": f"tiles sharded over {n_gpus} rank(s)"}


def run_reference_arm(args):
    """The reference algorithm on the host cores (oracle port).  Host only: the number does not depend on --gpus; for N > 1 it is
    extrapolated to the N-GPU arm's (larger) mosaic so that both arms state the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n, size, extent = mosaic_geometry(args.gpus)
    vals = []
    t_start = time.perf_counter()
    for i in range(args.warmup + args.steps):
        tps, ppm, sample = cpu_reference_sample(args.arch, threads, n_s=4 if args.arch == "vit_small" else 3)
        if i >= args.warmup:
            vals.append(cpu_value(tps, ppm, n * n, extent))
    v = statistics.mean(vals)
    mp = extent * extent / 1e6
    cfg = workload_config(args.arch, args.gpus, "f32 (torch CPU)", 1, 1)
    cfg["parallelism"] = f"host only ({threads} threads), independent of --gpus; stated on the workload of the {args.gpus}-GPU arm"
    cfg["note"] = "each step times a bounded sample and extrapolates linearly in tiles and pixels"
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "MP/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * mp / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": "MP/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": time.perf_counter() - t_start}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------- MIM pre-training step (configs[3])
def mim_flops_per_image(D, depth, heads, N, ldy=192):
    """2*M*N*K of every contraction, forward + input-gradient + weight-gradient (SURVEY.md 8d: 3 x (fwd 44.811 + decoder))."""
    K0 = 3 * PATCH * PATCH
    block = 2.0 * N * D * 3 * D + 4.0 * N * N * D + 2.0 * N * D * D + 4.0 * N * D * 4 * D
    fwd = 2.0 * (N - 1) * D * K0 + depth * block + 2.0 * N * D * ldy
    return 3.0 * fwd


def mim_cpu_sample(threads, batch=2, steps=1):
    """The reference training step (oracle port: torch-CPU autograd + restated clip / AdamW) on a bounded batch."""
    from oracle import train_oracle as TO
    from oracle import vit_oracle as VO
    torch.set_num_threads(threads)
    cfg = VO.ViTConfig(**ARCHS["vit_small"])
    sd = VO.init_state_dict(cfg, seed=0, mim=True)
    gd = torch.Generator().manual_seed(5)
    params = dict(sd)
    params["decoder.0.weight"], params["decoder.0.bias"] = torch.randn(192, cfg.embed_dim, 1, 1, generator=gd) * 0.02, torch.zeros(192)
    state = TO.TrainState(params)
    x = VO.synthetic_tile(WINDOW, seed=9, batch=batch)
    rs = np.random.RandomState(0)
    mask = torch.from_numpy(np.stack([VO.mask_generator(rs, WINDOW, 16, PATCH, 0.5) for _ in range(batch)]))
    t0 = time.perf_counter()
    for _ in range(steps):
        TO.train_step(state, cfg, x, mask)
    dt = time.perf_counter() - t0
    return batch * steps / dt, f"{steps} training step(s) of ViT-S/8 MIM at batch {batch} (224^2): torch-CPU fwd+bwd, clip 5.0, AdamW"



class Dist:
    """One process per GPU (torch.distributed over NCCL when WORLD_SIZE > 1)."""

    def __init__(self):
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.group = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.group = dist.group.WORLD

    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, v: float) -> float:
        t = torch.tensor([v], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    def bcast_obj(self, obj):
        if self.world == 1:
            return obj
        box = [obj]
        torch.distributed.broadcast_object_list(box, src=0)
        return box[0]

    def close(self):
        if self.world > 1:
            torch.distributed.barrier()
            torch.distributed.destroy_process_group()


def peak_tflops():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peaks = json.load(open(peaks_path))
        return float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0))), "measured (sustained cuBLAS bf16, MEASURED_PEAKS.json)"
    return 1400.0, "fallback (B200_PROFILING.md sustained figure)"


def kernel_source_hash(*names):
    h = hashlib.sha256()
    for n in names:
        with open(os.path.join(ROOT, "vit-ocm-wmsegmentation_b200", "csrc", n), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def ncu_traffic(kernel_class, key, scale):
    """DRAM bytes per launch from the committed ncu --set full capture (profiles/roofline_traffic.json) -- only while the kernel's
    source is the one that was captured (the record carries the source hash); otherwise null rather than a stale number."""
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if not os.path.exists(tpath):
        return None
    rec = json.load(open(tpath)).get(kernel_class)
    if not rec or key not in rec:
        return None
    files = rec.get("source_files")
    if not files or rec.get("source_sha16") != kernel_source_hash(*files):
        return None
    return rec[key] * scale


def mim_step(D, args, steps, warmup, with_e2e=True, sampler=None):
    """BASELINE.json configs[3]: MIM (SimMIM-style) pre-training step, ViT-S/8, 224^2 synthetic tiles, bf16 fwd+bwd with fp32
    master weights / AdamW, batch `batch_per_gpu` per GPU (32 -> 256 on 8), NCCL all-reduce of the flat gradient.  One step =
    zero_grad, forward, loss.sum().backward(), all-reduce, clip_grad_norm_(5.0), AdamW, bf16 weight repack.  -> dict of results."""
    import vitocm_b200 as vob
    from vitocm_b200 import synthetic as SY   # the GPU arm never touches oracle/
    from functools import partial
    from types import SimpleNamespace as NS
    world, rank, dev = D.world, D.rank, D.dev
    a = ARCHS["vit_small"]
    torch.manual_seed(0)
    enc = vob.VisionTransformerForSimMIM(patch_size=PATCH, embed_dim=a["embed_dim"], depth=a["depth"], num_heads=a["num_heads"], mlp_ratio=4,
                                         img_size=[WINDOW], qkv_bias=True, norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), precision="bf16")
    mim = vob.MIM(encoder=enc, encoder_stride=PATCH).cuda().train()
    cfg = NS(TRAIN=NS(BASE_LR=5e-4, WEIGHT_DECAY=0.05, CLIP_GRAD=5.0, OPTIMIZER=NS(NAME="adamw", EPS=1e-8, BETAS=(0.9, 0.999))))
    opt = vob.optimizer.build_pretrain_optimizer(cfg, mim, None)
    if world > 1:
        mim.overlap_grad_allreduce(True)     # every backward of this loop is final (no gradient accumulation)
    Bg = args.batch_per_gpu
    N = (WINDOW // PATCH) ** 2 + 1
    # a few distinct synthetic batches in pinned host memory (rank-dependent seeds), cycled through
    n_host = 4
    rs = np.random.RandomState(1000 + rank)
    base = SY.synthetic_tile(WINDOW, seed=500 + rank, batch=min(Bg, 8))
    xs_host = [base[torch.randint(0, base.shape[0], (Bg,), generator=torch.Generator().manual_seed(i))].contiguous().pin_memory() for i in range(n_host)]
    ms_host = [SY.random_masks(rs, Bg, WINDOW, 16, PATCH, 0.5).pin_memory() for _ in range(n_host)]
    xs_dev = [x.to(dev) for x in xs_host]
    ms_dev = [m.to(dev) for m in ms_host]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def train_step(x, m):
        opt.zero_grad()
        loss, _, _ = mim(x, m)
        loss.sum().backward()        # (the gradient all-reduce is launched from inside the backward, bucket by bucket)
        mim.all_reduce_grads()
        vob.optimizer.clip_grad_norm_(mim, cfg.TRAIN.CLIP_GRAD)
        opt.step()
        return loss

    for i in range(warmup):          # same cadence as the timed iterations (flush, barrier, step, barrier): the power-cap
        flush.fill_(1)               # controller then enters the timed region in its steady state
        D.barrier()
        train_step(xs_dev[i % n_host], ms_dev[i % n_host])
        D.barrier()
    if sampler is not None:
        sampler.open_window()
    launches0 = vob._lib.launch_count()
    step_ms = []
    for i in range(steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        D.barrier()
        e0.record()
        loss = train_step(xs_dev[i % n_host], ms_dev[i % n_host])
        e1.record()
        D.barrier()
        step_ms.append(e0.elapsed_time(e1))
    launches = vob._lib.launch_count() - launches0
    if sampler is not None:
        sampler.stop()
    ms_per_step = D.max_over_ranks(sum(step_ms)) / steps
    res = {"value": Bg * world / (ms_per_step / 1e3), "unit": "images/s", "ms_per_step": ms_per_step, "step_ms_rank0": [round(v, 3) for v in step_ms],
           "batch_per_gpu": Bg, "global_batch": Bg * world, "gpu_launches": int(launches)}
    if with_e2e:   # pinned host batch -> device inside the timed region, loss read back every step
        e2e_ms = []
        loss_host = torch.empty((), dtype=torch.float32).pin_memory()
        for i in range(2 + steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            D.barrier()
            e0.record()
            x = xs_host[i % n_host].to(dev, non_blocking=True)
            m = ms_host[i % n_host].to(dev, non_blocking=True)
            loss = train_step(x, m)
            loss_host.copy_(loss.detach(), non_blocking=True)
            e1.record()
            D.barrier()
            if i >= 2:
                e2e_ms.append(e0.elapsed_time(e1))
        e2e_t = D.max_over_ranks(sum(e2e_ms) / len(e2e_ms))
        res["e2e"] = {"value": Bg * world / (e2e_t / 1e3), "unit": "images/s",
                      "h2d_bytes_per_step": int(xs_host[0].numel() * 4 + ms_host[0].numel() * 8) * world, "d2h_bytes_per_step": 4 * world, "ms_per_step": e2e_t}
        res["final_loss"] = float(loss_host.item())
    # ---- per-kernel-class device times
    vob._lib.profile_enable(True)
    train_step(xs_dev[0], ms_dev[0])
    torch.cuda.synchronize()
    prof = vob._lib.profile_read()
    vob._lib.profile_enable(False)
    classes = {k: {"ms": v[0], "launches": v[1]} for k, v in prof.items() if v[1] > 0}
    Dm, depth = a["embed_dim"], a["depth"]
    M = Bg * N
    gemm_fwd = 2.0 * M * Dm * (3 * Dm + Dm + 8 * Dm) * depth
    attn_fwd = 4.0 * N * N * Dm * Bg * depth
    cls_gflop = {"gemm_wgrad": gemm_fwd + 2.0 * M * Dm * 192 * 2, "gemm_dgrad": gemm_fwd + 2.0 * M * Dm * 192, "attention": attn_fwd, "attention_bwd": 2.5 * attn_fwd,
                 "gemm_qkv": 2.0 * M * Dm * 3 * Dm * depth, "gemm_proj": 2.0 * M * Dm * Dm * depth, "gemm_fc1_gelu": 2.0 * M * Dm * 4 * Dm * depth,
                 "gemm_fc2": 2.0 * M * Dm * 4 * Dm * depth}
    for k, c in classes.items():
        c["gflop"] = cls_gflop.get(k, 0.0) / 1e9
        c["tflops"] = c["gflop"] / c["ms"] if c["ms"] > 0 and c["gflop"] > 0 else None
    peak, peak_src = peak_tflops()
    tensor_classes = {k: c for k, c in classes.items() if c["gflop"] > 0}
    dom = max(tensor_classes, key=lambda k: tensor_classes[k]["ms"])
    c = tensor_classes[dom]
    res["roofline"] = {"kernel": dom, "bound": "tensor", "achieved": c["tflops"], "peak": peak, "unit": "TFLOP/s", "frac": c["tflops"] / peak,
                       "traffic": ncu_traffic(dom, "dram_bytes_per_image_per_launch", Bg), "peak_source": peak_src,
                       "launches_per_step": c["launches"], "avg_launch_ms": c["ms"] / c["launches"]}
    gf = mim_flops_per_image(Dm, depth, a["num_heads"], N)
    step_tflops = gf * Bg / 1e12 / (ms_per_step / 1e3)
    res["step_tensor"] = {"tflops_per_gpu": step_tflops, "frac_of_peak": step_tflops / peak, "gflop_per_image": gf / 1e9}
    res["kernel_classes"] = classes
    del mim, opt, enc
    torch.cuda.empty_cache()
    return res


def main_mim(args):
    metric = "mim_pretrain_images_per_s"
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return
        threads = os.cpu_count() or 1
        vals = []
        for i in range(args.warmup + args.steps):
            ips, sample = mim_cpu_sample(threads, batch=2, steps=1)
            if i >= args.warmup:
                vals.append(ips)
        v = statistics.mean(vals)
        print(json.dumps({"impl": "reference", "metric": metric, "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": 1000.0 * args.batch_per_gpu * args.gpus / v, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": f"MIM pre-training step, vit_small/8, 224^2, global batch {args.batch_per_gpu * args.gpus}",
                                     "note": "host only; each step times a bounded batch-2 sample and extrapolates linearly in images"},
                          "cpu_baseline": {"value": v, "unit": "images/s", "cores": threads, "kind": "port", "sample": sample},
                          "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)
        return
    if args.warmup < 3:
        args.warmup = 3
    D = Dist()
    sampler = ClockSampler(D.local, enabled=D.rank == 0)
    sampler.start()
    r = mim_step(D, args, args.steps, args.warmup, with_e2e=True, sampler=sampler)
    if D.rank == 0:
        Bg = args.batch_per_gpu
        line = {"metric": metric, "value": r["value"], "unit": "images/s", "n_gpus": D.world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": r["ms_per_step"], "step_ms_rank0": r["step_ms_rank0"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16", "data": "synthetic",
                "config": {"workload": f"MIM pre-training step (SimMIM masked patches), vit_small/8, 224^2 synthetic tiles, batch {Bg} per GPU = {Bg * D.world} global, "
                                       "bf16 fwd+bwd, fp32 master weights + fused clip/AdamW, NCCL all-reduce(SUM) of the gradient buckets overlapped with the backward",
                           "batch_per_gpu": Bg, "global_batch": Bg * D.world, "weights": "random init (seed 0)",
                           "l2": "flushed between timed steps (256 MiB write, untimed); per-step working set >> L2",
                           "parallelism": f"data parallel over {D.world} rank(s)", "final_loss": r.get("final_loss")},
                "e2e": r["e2e"], "gpu_launches": r["gpu_launches"], "clocks": sampler.summary(), "roofline": r["roofline"],
                "step_tensor": r["step_tensor"], "kernel_classes": r["kernel_classes"]}
        if D.world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            ips, sample = mim_cpu_sample(threads)
            line["cpu_baseline"] = {"value": ips, "unit": "images/s", "cores": threads, "kind": "port", "sample": sample}
        print(json.dumps(line), flush=True)
    D.close()


# ------------------------------------------------------------------------------------- GPU arm
def time_segmentation(D, seg, mosaic, steps, warmup, flush, sampler=None, want=("th", "th3"), after_warmup=None):
    """`warmup` untimed + `steps` timed passes with the mosaic resident in HBM; CUDA events on the launching stream, barrier +
    synchronize on both sides of every step, L2 flushed in between.  -> (ms per step = max over ranks, rank-0 step list, last result)."""
    import gc
    gc.collect()                                         # (before the warm-up: an idle gap between warm-up and timed steps lets the GPU
    gc_was = gc.isenabled()                              #  boost and then be clamped: one timed step of 150-500 ms in one run of five)
    gc.disable()                                         # no collector pause between the launches of a step
    out = None
    prev = None
    extra = 0
    i = 0
    # warm-up: the requested steps, then (still untimed, at most 12 more) until two consecutive steps agree within 3 % on every rank --
    # after an idle phase the first steps run at ~1.93 GHz, then the power cap bites, and ONE step inside that transition reads 128 ms
    # against 70 (profiles/r02_gpu_call_al_final.log); the timed region must not start inside it
    while warmup > 0 and (i < warmup or extra < 12):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        D.barrier()
        e0.record()
        out = seg.segment(mosaic, want=want, gather=True)
        e1.record()
        D.barrier()
        cur = D.max_over_ranks(e0.elapsed_time(e1))
        i += 1
        settled = prev is not None and abs(cur - prev) <= 0.03 * prev
        prev = cur
        if i >= warmup:
            if settled:
                break
            extra += 1
    time_segmentation.extra_warmup = max(i - warmup, 0)
    if after_warmup is not None:
        after_warmup()
    if sampler is not None:
        sampler.open_window()
    step_ms = []
    D.barrier()
    for _ in range(steps):
        flush.fill_(1)                                   # evict L2 between timed steps (not timed)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        D.barrier()
        e0.record()
        out = seg.segment(mosaic, want=want, gather=True)
        e1.record()
        D.barrier()
        step_ms.append(e0.elapsed_time(e1))
    if gc_was:
        gc.enable()
    if sampler is not None:
        sampler.stop()
    return D.max_over_ranks(sum(step_ms)) / max(steps, 1), step_ms, out


def time_segmentation_e2e(D, seg, mosaic_host, host_masks, steps, warmup):
    """The same pass through the public API with HOST buffers: every rank uploads the rows of the pinned host mosaic it needs and
    copies its band of each mask into the shared pinned host image, all inside the timed region."""
    ms = []
    for i in range(warmup + steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        D.barrier()
        e0.record()
        seg.segment(mosaic_host, want=tuple(host_masks), gather=False, host_out=host_masks)
        e1.record()
        D.barrier()
        if i >= warmup:
            ms.append(e0.elapsed_time(e1))
    return D.max_over_ranks(sum(ms) / len(ms))


def shared_host_masks(D, vob, extent, names=("th", "th3"), tag="m"):
    """Page-locked host images [extent, extent] that every rank maps (one file per mask under /dev/shm for N > 1)."""
    if D.world == 1:
        return {k: torch.empty(extent, extent, dtype=torch.uint8).pin_memory() for k in names}, []
    paths = D.bcast_obj([f"/dev/shm/vitocm_bench_{os.getpid()}_{tag}_{k}" for k in names] if D.rank == 0 else None)
    masks = {}
    if D.rank == 0:
        for k, pth in zip(names, paths):
            masks[k] = vob.shared_pinned_u8(pth, (extent, extent), create=True)
    D.barrier()
    if D.rank != 0:
        for k, pth in zip(names, paths):
            masks[k] = vob.shared_pinned_u8(pth, (extent, extent), create=False)
    D.barrier()
    return masks, (paths if D.rank == 0 else [])


def release_host_masks(masks, paths):
    for t in masks.values():
        try:
            if not t.is_pinned() or paths:
                torch.cuda.cudart().cudaHostUnregister(t.data_ptr())
        except Exception:
            pass
    for pth in paths:
        try:
            os.unlink(pth)
        except OSError:
            pass


def masks_sha(out, names=("th", "th3")):
    h = hashlib.sha256()
    for k in names:
        h.update(out[k].cpu().numpy().tobytes())
    return h.hexdigest()[:16]


DUMP_SAMPLE = 1 << 22      # most elements written per output: 16 MiB in float32, so a whole dump stays below 64 MB


def dump_outputs(out, directory):
    """Writes what MosaicSegmenter.segment returned to the caller as <directory>/<name>.npy, so that two builds can be compared
    output for output: the masks th / th3, the per-tile low-res maps, the Otsu thresholds, the histograms and the min/max keys.
    Integer outputs are written as float64 (exact), the others as float32.  An output of more than DUMP_SAMPLE elements is
    represented by its elements at DUMP_SAMPLE distinct flat indices, drawn with seed 0 and sorted: the same indices for every
    run and build at a given mosaic size.  Smaller outputs are written whole, in their own shape."""
    os.makedirs(directory, exist_ok=True)
    for name in ("th", "th3", "lowres", "thresholds", "hists", "minmax_ord"):
        t = out[name]
        if t.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_SAMPLE, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        t = t.cpu()
        a = t.numpy().astype(np.float32 if t.is_floating_point() or t.dtype == torch.uint8 else np.float64)
        np.save(os.path.join(directory, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=6)   # the power cap needs ~5 steps to settle after an idle phase: a step inside the transition reads 128 ms against 70
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--arch", default="vit_small", choices=sorted(ARCHS))
    ap.add_argument("--precision", default="fp16", help="bf16 | fp16 | fp32, optionally +mlp2[:blocks] (vision_transformer.parse_precision)")
    ap.add_argument("--chunk-tiles", type=int, default=2048, help="most tiles per kernel launch (a rank's whole shard at the default)")
    ap.add_argument("--tile-batch", type=int, default=2048, help="most tiles per engine call")
    ap.add_argument("--lanes", type=int, default=1, help="chunks in flight on concurrent streams")
    ap.add_argument("--ingest", default="direct", choices=["direct", "crops"], help="segmentation: tiles read out of the uint8 mosaic by the patch embedding, or fp32 crops cut first")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip mask_agreement / precision_modes / cfg3 / mim_train / multi_gpu_bitwise_equal")
    ap.add_argument("--workload", default="segmentation", choices=["segmentation", "mim_train"],
                    help="segmentation = BASELINE.json configs[1] (the headline); mim_train = configs[3] (MIM pre-training step)")
    ap.add_argument("--batch-per-gpu", type=int, default=32, help="mim_train: images per GPU per step (256 over 8 GPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="segmentation: write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "segmentation" or args.impl != "ours"):
        ap.error("--dump-outputs writes the outputs of the GPU segmentation path (--workload segmentation --impl ours)")
    if args.workload == "mim_train":
        return main_mim(args)
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.warmup < 3:
        args.warmup = 3

    D = Dist()
    world, rank, dev = D.world, D.rank, D.dev
    import vitocm_b200 as vob
    from vitocm_b200 import synthetic as SY   # the GPU arm never touches oracle/

    def make_model(arch, precision):
        torch.manual_seed(0)               # identical random-init weights in every precision and on every rank
        return getattr(vob, arch)(patch_size=PATCH, num_classes=0, precision=precision, chunk_tiles=args.chunk_tiles, lanes=args.lanes).cuda().eval()

    a = ARCHS[args.arch]
    model = make_model(args.arch, args.precision)
    n, size, extent = mosaic_geometry(world)
    T = n * n
    N = (WINDOW // PATCH) ** 2 + 1
    mosaic_host = torch.from_numpy(SY.synthetic_mosaic_u8(size, seed=4321)).pin_memory()
    mosaic = mosaic_host.to(dev)
    seg = vob.MosaicSegmenter(model, window=WINDOW, stride=STRIDE, tile_batch=args.tile_batch, group=D.group, ingest=args.ingest)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    mp = extent * extent / 1e6

    sampler = ClockSampler(D.local, enabled=rank == 0)
    sampler.start()
    launches0 = None
    # warm-up first (same cadence as the timed steps), then count launches over the timed steps only
    # ONE call: the timed steps follow the warm-up without a gap (an idle gap of tens of ms lets the GPU boost, overshoot the power cap
    # and be clamped for a step: profiles/r02_gpu_call_am_an_bench_spread.log)
    mark = {}
    ms_per_step, step_ms, out = time_segmentation(D, seg, mosaic, args.steps, args.warmup, flush, sampler=sampler,
                                                  after_warmup=lambda: mark.__setitem__("l0", vob._lib.launch_count()))
    extra_warmup = getattr(time_segmentation, "extra_warmup", 0)
    launches = vob._lib.launch_count() - mark["l0"]
    value = mp / (ms_per_step / 1e3)
    if args.dump_outputs and rank == 0:      # before a later segment() call may reuse the buffers of `out`
        dump_outputs(out, args.dump_outputs)

    # ---- end to end through the public API with HOST buffers (pinned), copies inside the timed region
    host_masks, shm_paths = shared_host_masks(D, vob, extent)
    e2e_ms = time_segmentation_e2e(D, seg, mosaic_host, host_masks, args.steps, 2)
    e2e_value = mp / (e2e_ms / 1e3)
    r0, r1 = seg.mosaic_rows_needed(size)
    h2d = torch.tensor([float((r1 - r0) * size)], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(h2d)
    host_ok = None
    if rank == 0:     # the host images assembled by all ranks equal the masks gathered on the device
        host_ok = bool(all(torch.equal(host_masks[k], out[k].cpu()) for k in host_masks))

    # ---- per-kernel-class device times (CUDA events on the launching stream) for the roofline
    vob._lib.profile_enable(True)
    seg.segment(mosaic, want=("th", "th3"), gather=True)
    torch.cuda.synchronize()
    prof = vob._lib.profile_read()
    vob._lib.profile_enable(False)
    t0, t1 = vob.shard_range(T, rank, world)
    my_tiles = t1 - t0
    classes = {k: {"ms": v[0], "launches": v[1], "gflop": class_flops(k, a["embed_dim"], N, my_tiles, a["depth"]) / 1e9}
               for k, v in prof.items() if v[1] > 0}
    if "block_tail" in classes:
        # the block-tail kernel also computes the NEXT block's QKV projection: every QKV projection of the step that is not a launch of
        # the QKV GEMM class ran inside it (one engine call per chunk: launches per layer = launches of the block-tail class / (depth - 1))
        L = a["depth"] - 1
        per_layer = 2.0 * my_tiles * N * a["embed_dim"] * 3 * a["embed_dim"] / 1e9
        calls = max(classes["block_tail"]["launches"] // L, 1)
        qkv_launched = classes.get("gemm_qkv", {"launches": 0})["launches"] / calls      # layers whose QKV projection was a GEMM launch
        if "gemm_qkv" in classes:
            classes["gemm_qkv"]["gflop"] = per_layer * qkv_launched
        classes["block_tail"]["gflop"] += per_layer * (L - qkv_launched)
    for k, c in classes.items():
        c["tflops"] = (c["gflop"] / c["ms"]) if c["ms"] > 0 and c["gflop"] > 0 else None
    peak, peak_src = peak_tflops()
    tensor_classes = {k: c for k, c in classes.items() if c["gflop"] > 0}
    dom = max(tensor_classes, key=lambda k: tensor_classes[k]["ms"]) if tensor_classes else None
    roofline = None
    if dom:
        c = tensor_classes[dom]
        tiles_per_launch = my_tiles * (a["depth"] - 1) / max(c["launches"], 1)
        roofline = {"kernel": dom, "bound": "tensor", "achieved": c["tflops"], "peak": peak, "unit": "TFLOP/s",
                    "frac": c["tflops"] / peak, "traffic": ncu_traffic(dom, "dram_bytes_per_tile", tiles_per_launch), "peak_source": peak_src,
                    "launches_per_step": c["launches"], "avg_launch_ms": c["ms"] / c["launches"]}
    # the bandwidth-bound post-processing class against the HBM roofline (SURVEY.md 8d: 3 B per stitched pixel + 4 h w B per tile)
    hbm_roofline = None
    if "post" in classes:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        hbm_peak = float(json.load(open(peaks_path)).get("hbm_gbs", 6546.6)) if os.path.exists(peaks_path) else 6500.0
        y0, y1 = vob.shard_range(extent, rank, world)
        alg_bytes = 3.0 * (y1 - y0) * extent + 4.0 * (WINDOW // PATCH) ** 2 * T + 4.0 * a["num_heads"] * N * my_tiles
        ach = alg_bytes / 1e9 / (classes["post"]["ms"] / 1e3)
        hbm_roofline = {"kernel": "post (head_mean + stitch_gray/minmax/hist/mask + otsu)", "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                        "frac": ach / hbm_peak, "algorithmic_bytes": alg_bytes, "ms": classes["post"]["ms"], "launches": classes["post"]["launches"]}
    step_tflops = flops_per_tile(a["embed_dim"], a["depth"], a["num_heads"], N) * my_tiles / 1e12 / (ms_per_step / 1e3)
    clocks = sampler.summary()

    extras = {}
    if not args.no_extras:
        # ---- mask agreement of the headline precision against the fp32-parity mode (same mosaic, same weights, untimed)
        ref_model = make_model(args.arch, "fp32")
        ref_seg = vob.MosaicSegmenter(ref_model, window=WINDOW, stride=STRIDE, tile_batch=args.tile_batch, group=D.group, ingest=args.ingest)
        ref_out = ref_seg.segment(mosaic, want=("th", "th3"), gather=True)
        tiles_x = torch.cat([SY.synthetic_tile(WINDOW, seed=1234 if i == 0 else 100 + i, batch=1) for i in range(32)]).to(dev)

        def tile_agreement(m):
            got = vob.attention_masks(m, tiles_x)["masks"]
            ag = {}
            for i, k in ((0, "th"), (2, "th3")):
                v = (got[:, i] == tile_ref[:, i]).float().mean(dim=(1, 2))
                ag[k] = {"mean": float(v.mean()), "min": float(v.min()), "frac_tiles_ge_0.999": float((v >= 0.999).float().mean()), "config1_tile": float(v[0])}
            return ag

        tile_ref = vob.attention_masks(ref_model, tiles_x)["masks"]
        if rank == 0:
            extras["mask_agreement"] = {
                "against": "the fp32-parity mode (split-bf16, pinned to the reference at 4e-6 by tests/test_gpu_parity.py) on this GPU, same weights and inputs",
                "precision": args.precision,
                "mosaic": {k: float((out[k] == ref_out[k]).float().mean()) for k in ("th", "th3")},
                "tiles_224": tile_agreement(model), "n_tiles": 32, "bar": 0.999}
        # ---- other precision schedules on the same box (N = 1 only: short runs, same mosaic)
        if world == 1:
            modes = {}
            for prec in ("bf16", "fp16+mlp2", "fp32"):
                if prec == args.precision:
                    continue
                m2 = ref_model if prec == "fp32" else make_model(args.arch, prec)
                s2 = ref_seg if prec == "fp32" else vob.MosaicSegmenter(m2, window=WINDOW, stride=STRIDE, tile_batch=args.tile_batch, ingest=args.ingest)
                ms2, _, o2 = time_segmentation(D, s2, mosaic, 3, 2, flush)
                modes[prec] = {"value": mp / (ms2 / 1e3), "unit": "MP/s", "ms_per_step": ms2, "steps": 3, "warmup": 2,
                               "mask_agreement_mosaic": {k: float((o2[k] == ref_out[k]).float().mean()) for k in ("th", "th3")},
                               "mask_agreement_tiles_224": tile_agreement(m2)}
                if prec != "fp32":
                    del m2, s2
            extras["precision_modes"] = modes
        del ref_model, ref_seg, ref_out
        # ---- N > 1: the sharded result is bit-identical to one GPU doing everything
        if world > 1:
            same = None
            if rank == 0:
                solo = vob.MosaicSegmenter(model, window=WINDOW, stride=STRIDE, tile_batch=args.tile_batch, group=None, ingest=args.ingest)
                so = solo.segment(mosaic, want=("th", "th3"))
                same = bool(torch.equal(so["th"], out["th"]) and torch.equal(so["th3"], out["th3"]) and torch.equal(so["thresholds"], out["thresholds"]))
                del solo, so
            D.barrier()
            extras["multi_gpu_bitwise_equal"] = same
        del out
        torch.cuda.empty_cache()
        # ---- BASELINE configs[2]: ViT-B/8, fixed 16384^2 mosaic (21 025 tiles, extent 16 352^2), strong scaling
        extras["cfg3"] = run_cfg3(D, vob, SY, args, flush)
        torch.cuda.empty_cache()
        # ---- BASELINE configs[3]: MIM pre-training step at batch 32 per GPU
        r = mim_step(D, args, steps=5, warmup=3, with_e2e=True)
        r.pop("step_ms_rank0", None)
        r["config"] = "MIM pre-training step (SimMIM), vit_small/8, 224^2, batch 32 per GPU, bf16 fwd+bwd, fp32 master weights, fused clip + AdamW, NCCL all-reduce of gradient buckets overlapped with the backward"
        extras["mim_train"] = r

    if rank == 0:
        cfgd = workload_config(args.arch, world, args.precision, args.chunk_tiles, args.lanes)
        cfgd["tiles_per_gpu"] = my_tiles
        line = {"metric": METRIC, "value": value, "unit": "MP/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "extra_warmup_steps": int(extra_warmup),   # untimed steps beyond `warmup` until two consecutive steps agreed within 3 %
                "ms_per_step": ms_per_step, "step_ms_rank0": [round(v, 3) for v in step_ms], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": args.precision, "data": "synthetic", "config": cfgd,
                "tiles_per_s": T / (ms_per_step / 1e3),
                "e2e": {"value": e2e_value, "unit": "MP/s", "h2d_bytes_per_step": int(h2d.item()),
                        "d2h_bytes_per_step": int(2 * extent * extent), "ms_per_step": e2e_ms, "host_masks_match_device": host_ok,
                        "path": "MosaicSegmenter.segment(host mosaic, host_out=...): per-rank band upload, per-rank band download into one shared pinned image"},
                "gpu_launches": int(launches),
                "clocks": clocks,
                "roofline": roofline,
                "roofline_hbm": hbm_roofline,
                "step_tensor": {"tflops_per_gpu": step_tflops, "frac_of_peak": step_tflops / peak, "gflop_per_tile": flops_per_tile(a["embed_dim"], a["depth"], a["num_heads"], N) / 1e9},
                "kernel_classes": classes}
        line.update(extras)
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            tps, ppm, sample = cpu_reference_sample(args.arch, threads, n_s=3)
            line["cpu_baseline"] = {"value": cpu_value(tps, ppm, T, extent), "unit": "MP/s", "cores": threads, "kind": "port",
                                    "sample": sample, "tiles_per_s": tps}
        print(json.dumps(line), flush=True)
    release_host_masks(host_masks, shm_paths)
    D.close()


def run_cfg3(D, vob, SY, args, flush):
    """BASELINE.json configs[2]: ViT-B/8 sliding-window segmentation of a fixed 16384^2 mosaic (145^2 = 21 025 tiles, extent 16 352^2 =
    267.4 MP), tiles sharded over the ranks: STRONG scaling.  The mosaic is the 4096^2 synthetic field repeated 4 x 4.  Few steps
    (a step is seconds of ViT-B work); `mask_sha256_16` is the same string at every N when the result does not depend on the sharding."""
    size = 16384
    n = len(range(0, size - 2 * STRIDE, STRIDE))
    extent = (n - 1) * STRIDE + WINDOW
    mp = extent * extent / 1e6
    torch.manual_seed(0)
    model = vob.vit_base(patch_size=PATCH, num_classes=0, precision=args.precision, chunk_tiles=args.chunk_tiles).cuda().eval()
    base = torch.from_numpy(SY.synthetic_mosaic_u8(4096, seed=4321))
    mosaic_host = base.repeat(4, 4).contiguous().pin_memory()
    mosaic = mosaic_host.to(D.dev)
    seg = vob.MosaicSegmenter(model, window=WINDOW, stride=STRIDE, tile_batch=args.tile_batch, group=D.group, ingest=args.ingest)
    steps = 1 if D.world == 1 else 2
    ms, _, out = time_segmentation(D, seg, mosaic, steps, 1, flush)
    sha = masks_sha(out) if D.rank == 0 else None
    del out
    host_masks, paths = shared_host_masks(D, vob, extent, tag="c3")
    e2e_ms = time_segmentation_e2e(D, seg, mosaic_host, host_masks, 1, 1)
    r0, r1 = seg.mosaic_rows_needed(size)
    h2d = torch.tensor([float((r1 - r0) * size)], dtype=torch.float64, device=D.dev)
    if D.world > 1:
        torch.distributed.all_reduce(h2d)
    sha_host = None
    if D.rank == 0:
        hh = hashlib.sha256()
        for k in ("th", "th3"):
            hh.update(host_masks[k].numpy().tobytes())
        sha_host = hh.hexdigest()[:16]
    release_host_masks(host_masks, paths)
    T = n * n
    N = (WINDOW // PATCH) ** 2 + 1
    ab = ARCHS["vit_base"]
    tf = flops_per_tile(ab["embed_dim"], ab["depth"], ab["num_heads"], N) * T / 1e12 / (ms / 1e3) / D.world
    peak, _ = peak_tflops()
    res = {"workload": f"vit_base/8 sliding-window segmentation, {size}x{size} gray mosaic (4096^2 synthetic field repeated 4x4), window {WINDOW}, stride {STRIDE}, "
                       f"{T} tiles, extent {extent}^2, tiles sharded over {D.world} rank(s)", "scaling": "strong", "precision": args.precision,
           "value": mp / (ms / 1e3), "unit": "MP/s", "ms_per_step": ms, "steps": steps, "warmup": 1, "tiles_per_s": T / (ms / 1e3),
           "step_tflops_per_gpu": tf, "frac_of_peak": tf / peak,
           "e2e": {"value": mp / (e2e_ms / 1e3), "unit": "MP/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(h2d.item()), "d2h_bytes_per_step": int(2 * extent * extent)},
           "mask_sha256_16": sha, "mask_sha256_16_host_path": sha_host}
    del model, seg, mosaic
    return res


if __name__ == "__main__":
    main()
