"""Step rate of training with stochastic depth (drop_path_rate) against training without it.
    python tools/drop_path_bench.py [--out profiles/r06_drop_path.jsonl] [--steps K]
Prints the card's name, power limit and top SM clock, then, at batch 32 and 224^2 for ViT-S/8 (depth 12, 6 heads) and the
reference's encoder (D 384, 3 heads of 128, depth 4), in bf16 and fp16, the fine-tune step and the MIM step of
tools/encoder_grad_bench.py at drop_path_rate 0 and 0.1 (DINO's schedule over the blocks): images/s from CUDA events over K steps
after a warm-up, rate 0 and rate 0.1 alternating in three rounds in the same process, every round reported.
The expectation: rate 0 runs the launches of a build without drop path; rate 0.1 adds the draws of the scales, one copy of them into
the workspace, and one load per row in the proj / fc2 epilogues and in the LayerNorm backward.
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from encoder_grad_bench import finetune_rate, make_finetune  # noqa: E402
from mim_fp16_bench import B, IMG, MODELS, card, inputs, make_mim, step_rate  # noqa: E402

N_CLASSES = 1000
RATES = (0.0, 0.1)


def set_rate(enc, rate):
    """DINO's schedule (vit.py:155), as VisionTransformer(drop_path_rate=rate) sets it"""
    for blk, p in zip(enc.blocks, torch.linspace(0, rate, len(enc.blocks))):
        blk.drop_path.drop_prob = p.item()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    ap.add_argument("--steps", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("drop_path_bench needs a CUDA device")
    lines = []

    def emit(d):
        lines.append(d)
        print(json.dumps(d), flush=True)
    emit({"card": card(), "batch": B, "img": IMG, "head_classes": N_CLASSES, "rates": list(RATES)})
    x, mask = inputs(11)
    xc, mc = x.cuda(), mask.cuda()
    y = (torch.arange(B) % N_CLASSES).cuda()
    for model, (D, heads, depth) in MODELS.items():
        for prec in ("bf16", "fp16"):
            ft = make_finetune(D, heads, depth, prec)
            mim = make_mim(D, heads, depth, prec)[0]
            for rnd in range(3):
                for rate in RATES:
                    set_rate(ft[0], rate)
                    ms, ips = finetune_rate(ft, xc, y, a.steps)
                    emit({"model": model, "precision": prec, "round": rnd, "drop_path_rate": rate, "step": "finetune", "step_ms": ms,
                          "images_per_s": ips})
                for rate in RATES:
                    set_rate(mim.encoder, rate)
                    ms, ips = step_rate(mim, xc, mc, a.steps)
                    emit({"model": model, "precision": prec, "round": rnd, "drop_path_rate": rate, "step": "mim", "step_ms": ms,
                          "images_per_s": ips})
            del ft, mim
            torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(l) for l in lines) + "\n")


if __name__ == "__main__":
    main()
