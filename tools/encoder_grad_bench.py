"""Fine-tuning step rate of the encoder (vitocm_encoder_train_forward / vitocm_encoder_backward) next to the MIM step.
    python tools/encoder_grad_bench.py [--out FILE] [--steps K]
Prints the card's name, power limit and top SM clock, then, at batch 32 and 224^2 for ViT-S/8 (depth 12, 6 heads) and the
reference's encoder (D 384, 3 heads of 128, depth 4), in bf16 and fp16:
  - one fine-tune step -- zero_grad, forward_feats -> CLS row -> Linear head (1000 classes) -> cross-entropy -> backward ->
    torch.optim.AdamW over encoder + head -- and one MIM step (tools/mim_fp16_bench.py: forward, loss.sum().backward(),
    clip_grad_norm_, FusedAdamW): images/s from CUDA events over K steps after a warm-up, the two alternating in three rounds in the
    same process, every round reported;
  - one profiled fine-tune step per model and precision in a separate pass (vitocm_profile_enable): device ms and launches per
    kernel class, so the encoder backward's cost can be read against the MIM step's.
The expectation stated with the feature: about the MIM step's rate minus its decoder and loss.
"""
import argparse
import json
import os
import sys
from functools import partial

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import vitocm_b200 as vob  # noqa: E402
from mim_fp16_bench import B, IMG, MODELS, card, inputs, make_mim, step_rate  # noqa: E402
from oracle import vit_oracle as VO  # noqa: E402

N_CLASSES = 1000


def make_finetune(D, heads, depth, precision, seed=7):
    cfg = VO.ViTConfig(embed_dim=D, depth=depth, num_heads=heads, patch_size=8, img_size=IMG)
    sd = VO.randomize_affine(VO.init_state_dict(cfg, seed=seed), seed=seed + 1)
    enc = vob.VisionTransformer(img_size=[IMG], patch_size=8, embed_dim=D, depth=depth, num_heads=heads, mlp_ratio=4, qkv_bias=True,
                                norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), precision=precision)
    enc.load_state_dict(sd, strict=True)
    enc = enc.cuda().train()
    head = torch.nn.Linear(D, N_CLASSES).cuda()
    opt = torch.optim.AdamW(list(enc.parameters()) + list(head.parameters()), lr=1e-4, weight_decay=0.05)
    return enc, head, opt


def finetune_step(enc, head, opt, x, y):
    opt.zero_grad()
    loss = F.cross_entropy(head(enc.forward_feats(x)[:, 0]), y)
    loss.backward()
    opt.step()
    return loss


def finetune_rate(ft, x, y, steps, warm=3):
    for _ in range(warm):
        finetune_step(*ft, x, y)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        finetune_step(*ft, x, y)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return round(ms, 3), round(B / ms * 1e3, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    ap.add_argument("--steps", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("encoder_grad_bench needs a CUDA device")
    lines = []

    def emit(d):
        lines.append(d)
        print(json.dumps(d), flush=True)
    emit({"card": card(), "batch": B, "img": IMG, "head_classes": N_CLASSES})
    x, mask = inputs(11)
    xc, mc = x.cuda(), mask.cuda()
    y = (torch.arange(B) % N_CLASSES).cuda()
    for model, (D, heads, depth) in MODELS.items():
        for prec in ("bf16", "fp16"):
            ft = make_finetune(D, heads, depth, prec)
            mim = make_mim(D, heads, depth, prec)[0]
            for rnd in range(3):
                ms, ips = finetune_rate(ft, xc, y, a.steps)
                emit({"model": model, "precision": prec, "round": rnd, "step": "finetune", "step_ms": ms, "images_per_s": ips})
                ms, ips = step_rate(mim, xc, mc, a.steps)
                emit({"model": model, "precision": prec, "round": rnd, "step": "mim", "step_ms": ms, "images_per_s": ips})
            torch.cuda.synchronize()
            vob._lib.profile_read()          # drop anything recorded before
            vob._lib.profile_enable(True)
            finetune_step(*ft, xc, y)
            torch.cuda.synchronize()
            vob._lib.profile_enable(False)
            prof = {k: [round(v[0], 3), v[1]] for k, v in vob._lib.profile_read().items() if v[1]}
            emit({"model": model, "precision": prec, "step": "finetune", "profile_ms_launches": prof})
            del ft, mim
            torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(l) for l in lines) + "\n")


if __name__ == "__main__":
    main()
