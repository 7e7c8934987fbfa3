"""Images of different sizes through ViT-S/8: one call per image, one call per distinct size, and one varlen call, in one process.
    python tools/varlen_bench.py [--out FILE] [--images 256] [--reps 5] [--precision fp16]
ViT-S/8 (random-init weights of seed 0, as bench.py) on `--images` square gray images whose sides are drawn (seed 1234) from 128^2 to
512^2 in steps of 32 -- the spread of sizes of an evaluation set of ROIs that the reference runs one at a time (SSS/eval.py:126-136).
Three ways, alternating, `--reps` rounds of each after one untimed round:
  per_image: VisionTransformer.cls_attention_rows(x_i[None]) for every image;
  per_size:  one cls_attention_rows call per distinct size, on the stacked images of that size;
  varlen:    one cls_attention_rows_varlen call on the whole list.
Each round is timed with CUDA events around the whole list (inputs already on the device; no L2 flush: the inputs of one round,
~0.1 GB, are re-read from HBM by the next way anyway).  Reported per way: ms per round (median), images/s and algorithmic TFLOP/s
(bench.flops_per_tile at each image's own N, i.e. the per-block formula of SURVEY.md section 8d).  The varlen rows are checked
against the per-image rows, element for element, before timing.  The card's name and power limit are read in the same run.  One
JSON line per way is printed and appended to --out."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vitocm_b200 as vob  # noqa: E402
from bench import flops_per_tile  # noqa: E402

PATCH = 8


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--images", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--precision", default="fp16")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("varlen_bench needs a GPU")
    torch.manual_seed(0)
    model = vob.vit_small(patch_size=PATCH, num_classes=0, precision=args.precision).cuda().eval()
    rng = np.random.default_rng(1234)
    sides = [int(s) for s in rng.choice(np.arange(128, 513, 32), size=args.images)]
    g = torch.Generator(device="cuda").manual_seed(5)
    ims = [torch.rand(1, s, s, generator=g, device="cuda") for s in sides]
    by_size = {}
    for i, s in enumerate(sides):
        by_size.setdefault(s, []).append(i)
    stacks = {s: torch.stack([ims[i] for i in idx]) for s, idx in by_size.items()}
    D, depth, heads = model.embed_dim, len(model.blocks), model.num_heads
    gflop = sum(flops_per_tile(D, depth, heads, (s // PATCH) ** 2 + 1) for s in sides) / 1e9

    ways = {
        "per_image": lambda: [model.cls_attention_rows(x[None]) for x in ims],
        "per_size": lambda: [model.cls_attention_rows(x) for x in stacks.values()],
        "varlen": lambda: model.cls_attention_rows_varlen(ims),
    }
    ref = [model.cls_attention_rows(x[None])[0] for x in ims]
    got = model.cls_attention_rows_varlen(ims)
    bitwise = all(torch.equal(a, b) for a, b in zip(got, ref))
    for fn in ways.values():   # untimed round: module loads, workspaces, position tables
        fn()
    ms = {k: [] for k in ways}
    for _ in range(args.reps):
        for k, fn in ways.items():
            ms[k].append(timed(fn))
    dev = card()
    for k in ways:
        med = float(np.median(ms[k]))
        rec = dict(tool="varlen_bench", way=k, precision=args.precision, images=args.images, distinct_sizes=len(by_size),
                   tokens=int(sum((s // PATCH) ** 2 + 1 for s in sides)), ms_median=round(med, 3), ms_all=[round(v, 3) for v in ms[k]],
                   images_per_s=round(args.images / med * 1e3, 1), tflops_algorithmic=round(gflop / med, 1),
                   varlen_bitwise_equal_per_image=bitwise, device=dev)
        line = json.dumps(rec)
        print(line)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
