"""head_dim 64 against head_dim 128 at equal FLOPs: B = 32 tiles of N = 785 tokens, D = 384 as 6 heads x 64 and as 3 heads x 128.

    python tools/head_dim_bench.py [--out FILE]

Prints the card's name and power limit, then
  - attention forward (vitocm_attention, bf16 engine): device us per launch and TFLOP/s (4 B H N^2 dh per launch); head_dim 64 both
    through its default path (four-pipeline kernel + packed tails) and through the generic kernel alone (VITOCM_ATTN_QUAD=0, run in
    a child process because the library reads the knob once),
  - attention backward (vitocm_attention_bwd): device us and TFLOP/s (10 B H N^2 dh: S recomputed, dP, dV, dK, dQ),
  - one MIM step (zero_grad, forward, loss.sum().backward(), clip_grad_norm_ 5.0, AdamW) of build_model(args, depth=4,
    num_heads=3) -- the reference's encoder -- against depth=4, num_heads=6, batch 32 at 224^2: images/s.
Every time is CUDA events around many launches after a warm-up.  The attention operands (58 MB) fit the 126 MB L2 and are
re-read from there; both widths move the same bytes."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vitocm_b200 as vob  # noqa: E402
from vitocm_b200._lib import VitocmConfig, check, cur_stream, ptr  # noqa: E402

B, N, D = 32, 785, 384


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def engine(heads):
    dh = D // heads
    cfg = VitocmConfig(D, 1, heads, 4 * D, 8, 3, 1e-6, dh ** -0.5, 0)
    h = C.c_void_p()
    check(vob._lib.load_library().vitocm_create(C.byref(cfg), C.byref(h)))
    return h


def timed(fn, n, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3   # us


def attention(heads, backward=True):
    lib = vob._lib.load_library()
    dh = D // heads
    eng = engine(heads)
    g = torch.Generator(device="cuda").manual_seed(1)
    qkv = torch.randn(B * N, 3 * D, device="cuda", generator=g).to(torch.bfloat16)
    ctx = torch.empty(B * N, D, device="cuda", dtype=torch.bfloat16)
    st = cur_stream()
    fwd_us = timed(lambda: check(lib.vitocm_attention(eng, ptr(qkv), qkv.stride(0), B, N, ptr(ctx), ctx.stride(0), st)), 100)
    fwd_flops = 4.0 * B * heads * N * N * dh
    out = {"heads": heads, "head_dim": dh, "fwd_us": round(fwd_us, 1), "fwd_tflops": round(fwd_flops / fwd_us / 1e6, 1)}
    if backward:
        npad = (N + 127) // 128 * 128
        lse = torch.empty(B, heads, npad, device="cuda")
        check(lib.vitocm_attention_fwd_lse(eng, ptr(qkv), qkv.stride(0), B, N, ptr(ctx), ctx.stride(0), ptr(lse), st))
        dctx = (torch.randn(B * N, D, device="cuda", generator=g) * 0.5).to(torch.bfloat16)
        dqkv = torch.empty(B * N, 3 * D, device="cuda", dtype=torch.bfloat16)
        delta = torch.empty(B, heads, npad, device="cuda")
        dqacc = torch.zeros(B * N, D, device="cuda")
        bwd_us = timed(lambda: check(lib.vitocm_attention_bwd(eng, ptr(qkv), qkv.stride(0), ptr(ctx), ptr(dctx), dctx.stride(0), ptr(lse),
                                                               ptr(delta), ptr(dqacc), ptr(dqkv), dqkv.stride(0), B, N, st)), 50)
        out.update(bwd_us=round(bwd_us, 1), bwd_tflops=round(2.5 * fwd_flops / bwd_us / 1e6, 1))
    lib.vitocm_destroy(eng)
    return out


def mim(heads, steps=10, warm=3):
    from types import SimpleNamespace as NS
    from vitocm_b200 import synthetic as SY
    args = NS(MODEL=NS(PATCH_SIZE=8), DATA=NS(IMG_SIZE=224),
              TRAIN=NS(BASE_LR=5e-4, WEIGHT_DECAY=0.05, OPTIMIZER=NS(NAME="adamw", EPS=1e-8, BETAS=(0.9, 0.999))))
    torch.manual_seed(0)
    m = vob.MIM(encoder=vob.build_model(args, depth=4, num_heads=heads), encoder_stride=8).cuda().train()
    opt = vob.optimizer.build_pretrain_optimizer(args, m, None)
    x = SY.synthetic_tile(224, seed=5, batch=B).cuda()
    mask = SY.random_masks(np.random.RandomState(2), B, 224, 16, 8, 0.5).cuda()

    def step():
        opt.zero_grad()
        loss, _, _ = m(x, mask)
        loss.sum().backward()
        vob.optimizer.clip_grad_norm_(m, 5.0)
        opt.step()
    us = timed(step, steps, warm)
    return {"heads": heads, "head_dim": D // heads, "depth": 4, "batch": B, "step_ms": round(us / 1e3, 2), "images_per_s": round(B / us * 1e6, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    ap.add_argument("--generic64", action="store_true", help=argparse.SUPPRESS)   # child: head_dim 64 forward, generic kernel only
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("head_dim_bench needs a CUDA device")
    if a.generic64:
        print(json.dumps(attention(6, backward=False)))
        return
    lines = [{"card": card(), "shape": f"B={B} N={N} D={D}", "dtype": "bf16"}]
    for heads in (6, 3):
        lines.append({"attention": "default path", **attention(heads)})
    env = dict(os.environ, VITOCM_ATTN_QUAD="0")
    child = subprocess.run([sys.executable, os.path.abspath(__file__), "--generic64"], env=env, capture_output=True, text=True, check=True)
    lines.append({"attention": "generic kernel (VITOCM_ATTN_QUAD=0)", **json.loads(child.stdout.strip().splitlines()[-1])})
    for heads in (6, 3):
        lines.append({"mim_step": f"build_model(args, depth=4, num_heads={heads})", **mim(heads)})
    text = "\n".join(json.dumps(l) for l in lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
