"""MIM training in bf16 against fp16: step rate, gradient error against the float64 oracle, and the range of the fp16 backward.
    python tools/mim_fp16_bench.py [--out FILE] [--steps K]
Prints the card's name and power limit, then, at batch 32 and 224^2 for ViT-S/8 (depth 12, 6 heads) and the reference's encoder
(build_model(args, depth=4, num_heads=3): D 384, 3 heads of 128):
  - one MIM step (zero_grad, forward, loss.sum().backward(), clip_grad_norm_ 5.0, FusedAdamW) per precision: images/s from CUDA
    events over K steps after a warm-up; bf16 and fp16 alternate in three rounds in the same process and every round is reported,
  - the global relative L2 error of all parameter gradients of one step against oracle/train_oracle.py run in float64 on the device,
    both precisions on the same weights and inputs,
  - the loss-scaled fp16 backward's range: per block, the largest |value| and the share of non-zero values below 2^-14 (fp16's
    subnormals) of the tensors the backward stores in fp16 -- dA (the qkv and fc1-input gradients), dXb (the residual-stream
    gradient) and dXN (the LayerNorm-output and attention-output gradients) -- and of dY.  The values are the oracle's exact
    intermediate gradients times the loss scale S the device picks (same formula), read with autograd hooks on the oracle's Linears.
"""
import argparse
import json
import math
import os
import subprocess
import sys
from functools import partial
from types import SimpleNamespace as NS

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vitocm_b200 as vob  # noqa: E402
from oracle import train_oracle as TO  # noqa: E402
from oracle import vit_oracle as VO  # noqa: E402

B, IMG = 32, 224
LOSS_SCALE_K0 = 0   # train_kernels.cuh
MODELS = {"vit-small-depth12": (384, 6, 12), "reference-encoder": (384, 3, 4)}
ARGS = NS(MODEL=NS(PATCH_SIZE=8), DATA=NS(IMG_SIZE=IMG),
          TRAIN=NS(BASE_LR=5e-4, WEIGHT_DECAY=0.05, OPTIMIZER=NS(NAME="adamw", EPS=1e-8, BETAS=(0.9, 0.999))))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def inputs(seed):
    x = VO.synthetic_tile(IMG, seed=seed, batch=B)
    rs = np.random.RandomState(seed + 1)
    mask = torch.from_numpy(np.stack([VO.mask_generator(rs, IMG, 32, 8, 0.6) for _ in range(B)]))
    return x, mask


def make_mim(D, heads, depth, precision, seed=7):
    cfg = VO.ViTConfig(embed_dim=D, depth=depth, num_heads=heads, patch_size=8, img_size=IMG)
    sd = VO.randomize_affine(VO.init_state_dict(cfg, seed=seed, mim=True), seed=seed + 1)
    gd = torch.Generator().manual_seed(seed + 2)
    dec_w, dec_b = torch.randn(192, D, 1, 1, generator=gd) * 0.05, torch.randn(192, generator=gd) * 0.05
    enc = vob.VisionTransformerForSimMIM(patch_size=8, embed_dim=D, depth=depth, num_heads=heads, mlp_ratio=4, img_size=[IMG], qkv_bias=True,
                                         norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), precision=precision)
    enc.load_state_dict(sd, strict=True)
    mim = vob.MIM(encoder=enc, encoder_stride=8)
    mim.decoder[0].weight.data.copy_(dec_w)
    mim.decoder[0].bias.data.copy_(dec_b)
    params = dict(sd)
    params["decoder.0.weight"], params["decoder.0.bias"] = dec_w, dec_b
    return mim.cuda().train(), params, cfg


def step_rate(mim, x, mask, steps, warm=3):
    opt = vob.optimizer.build_pretrain_optimizer(ARGS, mim, None)

    def step():
        opt.zero_grad()
        loss, _, _ = mim(x, mask)
        loss.sum().backward()
        vob.optimizer.clip_grad_norm_(mim, 5.0)
        opt.step()
    for _ in range(warm):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return round(ms, 3), round(B / ms * 1e3, 1)


def grad_error(mim, ref):
    num = den = 0.0
    for n, p in mim.named_parameters():
        r = ref[n[len("encoder."):] if n.startswith("encoder.") else n]
        num += (p.grad.double() - r).pow(2).sum().item()
        den += r.pow(2).sum().item()
    return (num / den) ** 0.5


class Probe:
    """Autograd hooks on the oracle's Linears (per block: qkv, proj, fc1, fc2 in call order) and the decoder's 1 x 1 conv."""

    def __init__(self, depth):
        self.depth, self.calls, self.grads = depth, 0, []
        self.linear, self.conv2d = torch.nn.functional.linear, torch.nn.functional.conv2d

    def _keep(self, t, block, name):
        if t.requires_grad:
            t.register_hook(lambda g: self.grads.append((block, name, g.detach())))

    def _lin(self, x, w, b=None):
        y = self.linear(x, w, b)
        block, which = divmod(self.calls, 4)
        self.calls += 1
        role_out = {0: "dA", 1: "dXb", 2: "dA", 3: "dXb"}[which]
        self._keep(y, block, role_out)
        if which in (0, 1, 2):        # LayerNorm outputs (qkv, fc1) and the attention output (proj): dXN
            self._keep(x, block, "dXN")
        return y

    def _conv(self, x, w, b=None, *a, **k):
        y = self.conv2d(x, w, b, *a, **k)
        if x.requires_grad:           # the decoder (the patch embedding reads the image, which needs no gradient)
            self._keep(y, "head", "dY")
            self._keep(x, "head", "dXN")
        return y

    def __enter__(self):
        torch.nn.functional.linear, torch.nn.functional.conv2d = self._lin, self._conv
        return self

    def __exit__(self, *exc):
        torch.nn.functional.linear, torch.nn.functional.conv2d = self.linear, self.conv2d


def range_stats(params, cfg, x, mask):
    C, p = 3, cfg.patch_size
    coef = np.float32(1.0) / (np.float32(mask.double().sum().item() * p * p + 1e-5) * np.float32(C))
    _, ex = math.frexp(float(coef))
    S = 2.0 ** (LOSS_SCALE_K0 + 1 - ex)
    with Probe(cfg.depth) as pr:
        TO.mim_loss_and_grads(params, cfg, x, mask)
    rows = {}
    for block, name, g in pr.grads:
        v = (g.double() * S).abs().reshape(-1)
        nz = v[v > 0]
        r = rows.setdefault((str(block), name), [0.0, 0, 0])
        r[0] = max(r[0], v.max().item())
        r[1] += int((nz < 2.0 ** -14).sum().item())
        r[2] += int(nz.numel())
    out = [{"block": b, "tensor": n, "max_abs": float(f"{m:.4g}"), "share_below_2^-14": float(f"{s / max(c, 1):.3g}")}
           for (b, n), (m, s, c) in sorted(rows.items(), key=lambda kv: (kv[0][0] != "head", int(kv[0][0]) if kv[0][0] != "head" else 0, kv[0][1]))]
    top = max(r["max_abs"] for r in out)
    return S, out, top


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    ap.add_argument("--steps", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mim_fp16_bench needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    lines = [{"card": card(), "batch": B, "img": IMG}]

    def emit(d):
        lines.append(d)
        print(json.dumps(d), flush=True)
    print(json.dumps(lines[0]), flush=True)
    x, mask = inputs(11)
    xc, mc = x.cuda(), mask.cuda()
    for model, (D, heads, depth) in MODELS.items():
        mims = {prec: make_mim(D, heads, depth, prec) for prec in ("bf16", "fp16")}
        params, cfg = mims["bf16"][1], mims["bf16"][2]
        p64 = {k: v.double().cuda() for k, v in params.items()}
        ref_loss, ref = TO.mim_loss_and_grads(p64, cfg, x.double().cuda(), mc)
        for prec, (m, _, _) in mims.items():
            m.zero_grad(set_to_none=True)
            loss, _, _ = m(xc, mc)
            loss.sum().backward()
            emit({"model": model, "precision": prec, "loss": round(loss.item(), 6), "oracle_loss": round(ref_loss.item(), 6),
                  "grad_rel_l2_vs_float64": float(f"{grad_error(m, ref):.4g}")})
        del ref
        S, stats, top = range_stats(p64, cfg, x.double().cuda(), mc)
        emit({"model": model, "range": "fp16 backward, oracle intermediate gradients x S", "loss_scale_S": S, "k0": LOSS_SCALE_K0,
              "max_abs": top, "headroom_log2_below_65504": round(math.log2(65504.0 / top), 2)})
        for r in stats:
            emit({"model": model, **r})
        for rnd in range(3):
            for prec, (m, _, _) in mims.items():
                ms, ips = step_rate(m, xc, mc, a.steps)
                emit({"model": model, "precision": prec, "round": rnd, "step_ms": ms, "images_per_s": ips})
        del mims
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(l) for l in lines) + "\n")


if __name__ == "__main__":
    main()
