"""fp16 headroom of the encoder backward (vitocm_encoder_backward) from the float64 oracle: the largest |value * S| in each group
of 16-bit gradient tensors the backward forms, S = 2^e with max |dfeats| * S in [2^k0, 2^(k0 + 1)) (train_kernels.cuh,
LOSS_SCALE_K0), for the shapes and upstreams of tests/test_gpu_encoder_grad.py.  CPU only.

    python tools/encoder_grad_headroom.py [--k0 0]

Groups (TrainWs): dY = the seeded upstream d norm(x_l); dXb = the residual-stream gradient; dXN = d LayerNorm output and dCTX;
dA = dPRE (fc1 pre-activation) and dQKV.
"""
import argparse
import math
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from encoder_grad_cases import CASES, inputs, loss  # noqa: E402
from oracle import vit_oracle as VO  # noqa: E402


def _track(t, group, seen):
    t.retain_grad()
    seen.append((group, t))
    return t


def _feats(sd, cfg, x, n, seen):
    t = _track(VO.prepare_tokens(sd, cfg, x), "dXb", seen)
    outs = []
    for i in range(cfg.depth):
        pre = f"blocks.{i}."
        h = _track(VO._ln(t, sd[pre + "norm1.weight"], sd[pre + "norm1.bias"], cfg.eps), "dXN", seen)
        B, N, D = h.shape
        qkv = _track(F.linear(h, sd[pre + "attn.qkv.weight"], sd[pre + "attn.qkv.bias"]), "dA", seen)
        q, k, v = qkv.reshape(B, N, 3, cfg.num_heads, cfg.head_dim).permute(2, 0, 3, 1, 4)
        a = ((q @ k.transpose(-2, -1)) * cfg.head_dim ** -0.5).softmax(-1)
        ctx = _track((a @ v).transpose(1, 2).reshape(B, N, D), "dXN", seen)
        t = _track(t + F.linear(ctx, sd[pre + "attn.proj.weight"], sd[pre + "attn.proj.bias"]), "dXb", seen)
        h2 = _track(VO._ln(t, sd[pre + "norm2.weight"], sd[pre + "norm2.bias"], cfg.eps), "dXN", seen)
        p = _track(F.linear(h2, sd[pre + "mlp.fc1.weight"], sd[pre + "mlp.fc1.bias"]), "dA", seen)
        t = _track(t + F.linear(F.gelu(p), sd[pre + "mlp.fc2.weight"], sd[pre + "mlp.fc2.bias"]), "dXb", seen)
        if cfg.depth - i <= n:
            outs.append(_track(VO._ln(t, sd["norm.weight"], sd["norm.bias"], cfg.eps), "dY", seen))
    return outs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--k0", type=int, default=0)
    args = ap.parse_args()
    for case, (cfg, H, W, B) in CASES.items():
        sd = {k: v.double().requires_grad_(True) for k, v in VO.randomize_affine(VO.init_state_dict(cfg, seed=21), seed=22).items()}
        x, u = inputs(cfg, H, W, B, seed=23)
        x = x.double()
        for upstream in ("head", "feats", "intermediate"):
            seen = []
            with torch.enable_grad():
                loss_v = loss(upstream, lambda: _feats(sd, cfg, x, 1, seen)[0], lambda: _feats(sd, cfg, x, 1, seen)[0][:, 0],
                             lambda: _feats(sd, cfg, x, 4, seen), u, torch.float64, "cpu")
                loss_v.backward()
            amax = max(t.grad.abs().max().item() for g, t in seen if g == "dY")
            S = 2.0 ** (args.k0 + 1 - math.frexp(amax)[1])
            peak = {}
            for g, t in seen:
                if t.grad is not None:
                    peak[g] = max(peak.get(g, 0.0), t.grad.abs().max().item() * S)
            print(f"{case:18s} {upstream:12s} S=2^{int(math.log2(S)):+d}  " +
                  "  ".join(f"{g} {peak.get(g, 0.0):.3g}" for g in ("dY", "dXb", "dXN", "dA")) +
                  f"  headroom 2^{math.log2(65504 / max(peak.values())):.1f}")


if __name__ == "__main__":
    main()
