"""Shapes, inputs and upstream losses of the encoder fine-tuning checks (tests/test_gpu_encoder_grad.py) and of the fp16 headroom
tool (tools/encoder_grad_headroom.py), with the float64 functional forward they are compared against.  No GPU, no pytest."""
import torch
import torch.nn.functional as F

from oracle import vit_oracle as VO

CASES = {
    # ViT-S/8 at 224^2, batch 2; the reference's MIM encoder (D 384, 3 heads of 128, depth 4), batch 8; a tiny model on a 48 x 64
    # input, whose position table is the bicubic resize of the 28 x 28 one
    "vit-small": (VO.ViTConfig(embed_dim=384, depth=12, num_heads=6), 224, 224, 2),
    "reference-encoder": (VO.ViTConfig(embed_dim=384, depth=4, num_heads=3), 224, 224, 8),
    "tiny-48x64": (VO.ViTConfig(embed_dim=128, depth=3, num_heads=2), 48, 64, 4),
}
N_CLASSES = 10


def inputs(cfg, H, W, B, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 3, H, W, generator=g)
    N = (H // cfg.patch_size) * (W // cfg.patch_size) + 1
    head_w = torch.randn(N_CLASSES, cfg.embed_dim, generator=g) * 0.2
    head_b = torch.randn(N_CLASSES, generator=g) * 0.1
    labels = torch.randint(0, N_CLASSES, (B,), generator=g)
    r_feats = torch.randn(B, N, cfg.embed_dim, generator=g)
    r_inter = torch.randn(B, min(4, cfg.depth) * cfg.embed_dim, generator=g)   # n > depth gives every block, as the reference
    return x, dict(head_w=head_w, head_b=head_b, labels=labels, r_feats=r_feats, r_inter=r_inter)


def loss(upstream, feats_fn, fwd_fn, inter_fn, u, dt, dev):
    """The three upstreams: forward -> linear head -> cross-entropy; forward_feats . fixed tensor; get_intermediate_layers(n=4)
    CLS rows concatenated . fixed tensor."""
    if upstream == "head":
        logits = F.linear(fwd_fn(), u["head_w"].to(dev, dt), u["head_b"].to(dev, dt))
        return F.cross_entropy(logits, u["labels"].to(dev))
    if upstream == "feats":
        return (feats_fn() * u["r_feats"].to(dev, dt)).sum()
    return (torch.cat([f[:, 0] for f in inter_fn()], dim=-1) * u["r_inter"].to(dev, dt)).sum()


def oracle_feats(sd, cfg, x, n):
    """get_intermediate_layers (vit.py:248-256) over oracle/vit_oracle.py's functional pieces, differentiable."""
    t = VO.prepare_tokens(sd, cfg, x)
    outs = []
    for i in range(cfg.depth):
        t, _, _ = VO.block(sd, cfg, i, t)
        if cfg.depth - i <= n:
            outs.append(VO._ln(t, sd["norm.weight"], sd["norm.bias"], cfg.eps))
    return outs
