"""Drop-in for the MIM half of the reference's ``model.py`` on B200 (forward / loss evaluation).

Mirrors ``VisionTransformerForSimMIM`` (SSS/model.py:11-53), ``MIM`` (:55-89) and ``build_model``
(:91-108): same constructor arguments, parameter names (``mask_token``, ``decoder.0.{weight,bias}``) and
return values.  The arithmetic runs in libvitocm.so (``vitocm_mim_forward``): patch-embedding GEMM with the
mask-token mix fused in its epilogue, the transformer blocks, final norm, the 1x1-conv decoder as a
per-token tcgen05 GEMM, PixelShuffle + masked L1 in one pass.

Training (SSS/mim.py:153-182): when gradients are enabled and a parameter requires them, ``MIM.forward`` runs
``vitocm_mim_train_forward`` inside a ``torch.autograd.Function`` whose backward is ``vitocm_mim_backward`` --
``loss.sum().backward()``, ``clip_grad_norm_`` and ``optimizer.step()`` of the reference loop work unchanged.  All
parameters then live in one flat fp32 buffer and their ``.grad`` in another (``MIM.flatten_parameters``), which is what
the fused clip + AdamW kernel (``optimizer.FusedAdamW``) and the NCCL gradient all-reduce operate on.
``MaskGenerator`` (SSS/data.py:163-186) is host-side numpy in the reference and stays so.
"""
from __future__ import annotations

import math
from functools import partial

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from ._lib import check, cur_stream, ptr
from .vision_transformer import VisionTransformer


class MaskGenerator:
    """SSS/data.py:163-186 (uses numpy's global RNG, like the reference)."""

    def __init__(self, input_size=192, mask_patch_size=32, model_patch_size=4, mask_ratio=0.6):
        assert input_size % mask_patch_size == 0 and mask_patch_size % model_patch_size == 0
        self.input_size, self.mask_patch_size, self.model_patch_size, self.mask_ratio = input_size, mask_patch_size, model_patch_size, mask_ratio
        self.rand_size = input_size // mask_patch_size
        self.scale = mask_patch_size // model_patch_size
        self.token_count = self.rand_size ** 2
        self.mask_count = int(np.ceil(self.token_count * mask_ratio))

    def __call__(self):
        idx = np.random.permutation(self.token_count)[:self.mask_count]
        mask = np.zeros(self.token_count, dtype=int)
        mask[idx] = 1
        return mask.reshape(self.rand_size, self.rand_size).repeat(self.scale, axis=0).repeat(self.scale, axis=1)


class VisionTransformerForSimMIM(VisionTransformer):
    """SSS/model.py:11-53.  As in the reference, ``img_size`` is *not* forwarded to the base constructor (the
    position table always has 28*28+1 rows for patch 8) and is bicubically resized whenever img_size[0] != 224."""

    def __init__(self, interpolate_encoding=False, img_size=224, **kwargs):
        super().__init__(**kwargs)
        self.mask_token = nn.Parameter(torch.zeros(1, 1, self.embed_dim))
        self.img_size = img_size
        self._trunc_normal_(self.mask_token, std=.02)
        self.interpolate_encoding = interpolate_encoding

    def _trunc_normal_(self, tensor, mean=0., std=1.):
        cdf = lambda v: (1.0 + math.erf(v / math.sqrt(2.0))) / 2.0   # noqa: E731  (a = -std, b = std)
        lo, hi = cdf(-1.0), cdf(1.0)
        with torch.no_grad():
            tensor.uniform_(2 * lo - 1, 2 * hi - 1).erfinv_().mul_(std * math.sqrt(2.0)).add_(mean).clamp_(min=-std, max=std)
        return tensor

    def _mim_pos_args(self, x):
        """(npatch, w, h) of the position table for input x: resized to img_size when that is not 224."""
        size = self.img_size[0] if isinstance(self.img_size, (list, tuple)) else self.img_size
        B, _, H, W = x.shape
        n = (H // self.patch_embed.patch_size) * (W // self.patch_embed.patch_size)
        if size != 224:
            return n, size, size
        return self.pos_embed.shape[1] - 1, 224, 224

    def _mim_pos(self, x):
        return self._pos_table(*self._mim_pos_args(x))

    @torch.no_grad()
    def forward(self, x, mask):
        """-> [B, D, H/p, W/p] (model.py:25-53)."""
        assert mask is not None
        xx = self._check_input(x)
        eng = self._ensure_engine()
        B, _, H, W = xx.shape
        N = self._tokens(xx)
        pos = self._mim_pos(xx)
        assert pos.shape[0] == N, "position table does not match the token count (img_size vs input size)"
        X = torch.empty(B, N, self.embed_dim, dtype=torch.float32, device=xx.device)
        m = mask.detach().reshape(B, -1).to(device=xx.device, dtype=torch.float32).contiguous()
        check(_lib.load_library().vitocm_prepare_tokens(eng, ptr(xx), B, H, W, ptr(pos), ptr(m), ptr(X), cur_stream()))
        self._run_blocks(X, 0, self.depth)
        z = self._final_norm(X)[:, 1:]
        h = w = int((N - 1) ** 0.5)
        return z.permute(0, 2, 1).reshape(B, self.embed_dim, h, w)     # a view change, no arithmetic

    # NB: like the reference's encoder (SSS/model.py:11-53, vit.py:135-258) this class has no ``no_weight_decay``: the
    # skip list of build_pretrain_optimizer is empty and cls_token / pos_embed / mask_token (3-D) do get weight decay.


class _MIMStep(torch.autograd.Function):
    """loss = MIM(x, mask) with the backward of SSS/mim.py:174 in libvitocm.  Parameter gradients do not travel through
    autograd: vitocm_mim_backward accumulates them straight into the flat ``.grad`` buffer of ``MIM`` (the parameters are
    passed as inputs only so that autograd schedules this node); the position table's gradient is returned."""

    @staticmethod
    def forward(ctx, mim, xx, maskf, pos, *params):
        enc = mim.encoder
        eng = enc._ensure_engine()
        lib = _lib.load_library()
        B, C, H, W = xx.shape
        N = enc._tokens(xx)
        x_rec = torch.empty_like(xx)
        sums = torch.empty(2, dtype=torch.float64, device=xx.device)
        need = int(lib.vitocm_mim_train_workspace_bytes(eng, B, N))
        if mim._train_ws is None or mim._train_ws.numel() < need or mim._train_ws.device != xx.device:
            mim._train_ws = None
            mim._train_ws = torch.empty(need, dtype=torch.uint8, device=xx.device)
        posc = pos.detach().to(torch.float32).contiguous()
        check(lib.vitocm_mim_train_forward(eng, ptr(xx), B, H, W, ptr(posc), ptr(maskf), ptr(x_rec), ptr(sums), ptr(mim._train_ws),
                                           mim._train_ws.numel(), cur_stream()))
        ctx.mim = mim
        # the saved activations live in the ONE shared workspace: stamp it, so that a backward whose forward has since been
        # overwritten by another training-mode forward fails loudly instead of producing wrong gradients
        mim._train_ws_gen = getattr(mim, "_train_ws_gen", 0) + 1
        ctx.ws_gen = mim._train_ws_gen
        ctx.save_for_backward(xx, maskf, x_rec, sums)
        ctx.pos_shape = tuple(pos.shape)
        ctx.mark_non_differentiable(x_rec)
        loss = (sums[0] / (sums[1] + 1e-5) / mim.in_chans).to(torch.float32)
        return loss, x_rec

    @staticmethod
    def backward(ctx, grad_loss, _grad_xrec):
        mim = ctx.mim
        if ctx.ws_gen != getattr(mim, "_train_ws_gen", 0):
            raise _lib.VitocmError("MIM backward: the activations of this forward were overwritten by a later training-mode forward "
                                   "(call backward() before the next forward, or run evaluation under model.eval())")
        xx, maskf, x_rec, sums = ctx.saved_tensors
        B, C, H, W = xx.shape
        mim._prepare_grads()
        dpos = torch.empty(ctx.pos_shape, dtype=torch.float32, device=xx.device)
        gs = grad_loss.detach().to(torch.float32).reshape(1).contiguous()      # stays on the device: no host sync
        check(_lib.load_library().vitocm_mim_backward(mim.encoder._engine, ptr(xx), B, H, W, ptr(maskf), ptr(x_rec), ptr(sums), ptr(gs),
                                                      ptr(dpos), ptr(mim._train_ws), mim._train_ws.numel(), cur_stream()))
        mim._launch_bucket_allreduce()
        return (None, None, None, dpos) + (None,) * len(mim._param_list)


class MIM(nn.Module):
    """SSS/model.py:55-89: encoder + (1x1 conv, PixelShuffle) decoder + masked L1 loss."""

    def __init__(self, encoder, encoder_stride):
        super().__init__()
        self.encoder = encoder
        self.encoder_stride = encoder_stride
        self.decoder = nn.Sequential(
            nn.Conv2d(in_channels=self.encoder.num_features, out_channels=self.encoder_stride ** 2 * 3, kernel_size=1),
            nn.PixelShuffle(self.encoder_stride),
        )
        self.in_chans = 3
        self.patch_size = 8
        if encoder_stride != encoder.patch_embed.patch_size:
            raise NotImplementedError("vitocm MIM: encoder_stride must equal the patch size")
        # the decoder's parameters are loaded into the encoder's engine under their state-dict names
        self.encoder._extra_engine_params = lambda: [("decoder.0.weight", self.decoder[0].weight), ("decoder.0.bias", self.decoder[0].bias)]
        self._train_ws = None
        self._param_list = None      # [(engine name, parameter)] in flat-buffer order
        self._pflat = self._gflat = None
        self._grad_views = None
        self._flat_ptrs = None
        self._overlap_group = None   # overlap_grad_allreduce(): process group (or True = WORLD) for the bucketed all-reduce
        self._overlap = False
        self._comm_stream = None
        self._comm_done = None       # event: the bucket all-reduces of the last backward have finished
        self._bwd_events = None

    # ------------------------------------------------------------------ training plumbing
    def _engine_name(self, pname: str) -> str:
        return pname[len("encoder."):] if pname.startswith("encoder.") else pname

    def flatten_parameters(self):
        """Move every parameter into one flat fp32 device buffer (``self._pflat``) and give it a ``.grad`` view into a
        second one (``self._gflat``): the engine aliases the weights (vitocm_bind_weight), the backward kernels accumulate
        straight into the gradients (vitocm_bind_grad), and clip / AdamW / the NCCL all-reduce are single flat operations.
        Offsets are 16-byte aligned.  Idempotent; call after ``.cuda()``."""
        named = [(n, p) for n, p in self.named_parameters() if p.requires_grad]
        dev = named[0][1].device
        if dev.type != "cuda":
            raise _lib.VitocmError("vitocm MIM training needs the parameters on a CUDA device (no CPU path)")
        ptrs = tuple(p.data_ptr() for _, p in named)
        if self._pflat is not None and ptrs == self._flat_ptrs:
            return self
        offs, total = [], 0
        for _, p in named:
            offs.append(total)
            total += (p.numel() + 3) // 4 * 4
        pflat = torch.zeros(total, dtype=torch.float32, device=dev)
        gflat = torch.zeros(total, dtype=torch.float32, device=dev)
        views = []
        with torch.no_grad():
            for (n, p), o in zip(named, offs):
                pflat[o:o + p.numel()].copy_(p.detach().reshape(-1).to(torch.float32))
                p.data = pflat[o:o + p.numel()].view(p.shape)
                g = gflat[o:o + p.numel()].view(p.shape)
                if p.grad is not None:
                    g.copy_(p.grad)
                p.grad = g
                views.append(g)
        self._pflat, self._gflat, self._grad_views, self._flat_offsets = pflat, gflat, views, offs
        self._param_list = [(self._engine_name(n), p) for n, p in named]
        self._flat_ptrs = tuple(p.data_ptr() for _, p in named)
        self.encoder._grads_bound_to = None
        self.encoder._bind_weights = True
        return self

    def decay_flags(self, skip_list=(), skip_keywords=()):
        """uint8 [numel of the flat buffer]: 1 where AdamW applies weight decay -- the has_decay / no_decay split of
        get_pretrain_param_groups (SSS/optimizer.py:14-33): none for 1-D parameters, biases, and the skip list."""
        self.flatten_parameters()
        flags = torch.zeros(self._pflat.numel(), dtype=torch.uint8, device=self._pflat.device)
        for (n, p), o in zip([(n, p) for n, p in self.named_parameters() if p.requires_grad], self._flat_offsets):
            no_decay = len(p.shape) == 1 or n.endswith(".bias") or n in skip_list or any(k in n for k in skip_keywords)
            if not no_decay:
                flags[o:o + p.numel()] = 1
        return flags

    def _prepare_grads(self):
        """Before a backward: every parameter's ``.grad`` must be its view into the flat buffer.  After
        ``optimizer.zero_grad()`` (set_to_none) the views are re-attached and the buffer is zeroed (one memset)."""
        self.flatten_parameters()
        none = [p.grad is None for _, p in self._param_list]
        if all(none):
            self._gflat.zero_()
            for (_, p), g in zip(self._param_list, self._grad_views):
                p.grad = g
        elif any(none) or any(p.grad is not g for (_, p), g in zip(self._param_list, self._grad_views)):
            for (_, p), g in zip(self._param_list, self._grad_views):     # mixed state: keep what is there, re-home it
                if p.grad is None:
                    g.zero_()
                elif p.grad is not g:
                    g.copy_(p.grad)
                p.grad = g
        eng = self.encoder._engine
        # the binding cache lives on the encoder: a differentiable encoder call on the same engine rebinds to its own buffers
        key = ("mim", eng.value, self._gflat.data_ptr())
        if self.encoder._grads_bound_to != key:
            lib = _lib.load_library()
            for (name, p), g in zip(self._param_list, self._grad_views):
                if name != "pos_embed":
                    check(lib.vitocm_bind_grad(eng, name.encode(), g.data_ptr()))
            self.encoder._grads_bound_to = key

    def overlap_grad_allreduce(self, enabled: bool = True, group=None):
        """Data-parallel training: launch the gradient all-reduce from INSIDE the next backward(s), one bucket per transformer
        block (plus one for decoder + final norm), each as soon as that block's gradients are complete
        (vitocm_mim_backward_events), on a side stream -- the collectives then run under the rest of the backward instead of
        after it.  ``all_reduce_grads()`` afterwards only reduces the small embedding bucket (its pos_embed part is accumulated by
        autograd after the backward kernel sequence) and joins the side stream.  Enable it only for a backward whose gradient is
        final (the LAST micro-step under gradient accumulation): reducing a partial sum twice would count it R times."""
        self._overlap = bool(enabled)
        self._overlap_group = group
        return self

    def _buckets(self):
        """[(event index, flat begin, flat end)] in backward order + the embedding range: blocks l own a contiguous range of the
        flat buffer (named_parameters order), decoder + final norm the tail, cls / pos / mask token / patch filter the head."""
        names = [n for n, _ in self._param_list]
        offs = list(self._flat_offsets) + [self._pflat.numel()]
        depth = self.encoder.depth

        def span(pred):
            idx = [i for i, n in enumerate(names) if pred(n)]
            assert idx == list(range(idx[0], idx[-1] + 1)), "parameters of one bucket must be contiguous in the flat buffer"
            return offs[idx[0]], offs[idx[-1] + 1]

        out = [(depth,) + span(lambda n: n.startswith("norm.") or n.startswith("decoder."))]
        for l in range(depth - 1, -1, -1):
            out.append((l,) + span(lambda n, l=l: n.startswith(f"blocks.{l}.")))
        embed = span(lambda n: not (n.startswith("blocks.") or n.startswith("norm.") or n.startswith("decoder.")))
        return out, embed

    def _launch_bucket_allreduce(self):
        """Called by the backward right after vitocm_mim_backward has enqueued its kernels."""
        import torch.distributed as dist
        self._comm_done = None
        if not self._overlap or not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(self._overlap_group) < 2:
            return
        lib = _lib.load_library()
        eng = self.encoder._engine
        depth = self.encoder.depth
        if self._bwd_events is None or self._bwd_events[0] != eng.value:
            import ctypes as C
            arr = (C.c_void_p * (depth + 1))()
            check(lib.vitocm_mim_backward_events(eng, arr, depth + 1))
            self._bwd_events = (eng.value, [arr[i] for i in range(depth + 1)])
            # the events only exist from now on: this first backward was not instrumented -> flat reduce in all_reduce_grads()
            return
        if self._comm_stream is None:
            self._comm_stream = torch.cuda.Stream()
        buckets, _ = self._buckets()
        with torch.cuda.stream(self._comm_stream):
            for ev_idx, lo, hi in buckets:
                check(lib.vitocm_stream_wait_event(self._comm_stream.cuda_stream, self._bwd_events[1][ev_idx]))
                dist.all_reduce(self._gflat[lo:hi], op=dist.ReduceOp.SUM, group=self._overlap_group)
            self._comm_done = torch.cuda.Event()
            self._comm_done.record(self._comm_stream)

    def all_reduce_grads(self, group=None):
        """Data parallelism over one process per GPU: sum the gradients across ranks (NCCL over NVLink).
        The reference trains under nn.DataParallel with ``loss.sum().backward()`` (SSS/mim.py:102,174): the gradient is
        the SUM over replicas of each replica's mean loss, which is exactly all_reduce(SUM) of the per-rank gradients.
        Order: backward -> all_reduce_grads -> clip_grad_norm_ -> optimizer.step.  After a backward that ran with
        ``overlap_grad_allreduce`` only the embedding bucket is left to reduce; otherwise the whole flat buffer is."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1):
            return
        if self._comm_done is not None:
            _, (lo, hi) = self._buckets()
            dist.all_reduce(self._gflat[lo:hi], op=dist.ReduceOp.SUM, group=group)
            torch.cuda.current_stream().wait_event(self._comm_done)
            self._comm_done = None
        else:
            dist.all_reduce(self._gflat, op=dist.ReduceOp.SUM, group=group)

    def _forward_train(self, x, mask):
        enc = self.encoder
        self.flatten_parameters()
        xx = enc._check_input(x)
        B = xx.shape[0]
        N = enc._tokens(xx)
        pos = enc._pos_graph(*enc._mim_pos_args(xx))
        assert pos.shape[0] == N, "position table does not match the token count (img_size vs input size)"
        m = mask.detach().reshape(B, -1).to(device=xx.device, dtype=torch.float32).contiguous()
        loss, x_rec = _MIMStep.apply(self, xx, m, pos, *[p for _, p in self._param_list])
        mask_up = mask.repeat_interleave(self.patch_size, 1).repeat_interleave(self.patch_size, 2).unsqueeze(1).contiguous()
        return loss, x_rec, mask_up

    def forward(self, x, mask):
        """-> (loss, x_rec, mask upsampled to pixels) (model.py:71-77).  With gradients enabled the loss carries the
        backward of the training step (``model.train()``, as SSS/mim.py:154 sets it); in ``eval()`` mode or under
        ``torch.no_grad()`` this is a plain evaluation."""
        if self.training and torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            return self._forward_train(x, mask)
        return self._forward_eval(x, mask)

    @torch.no_grad()
    def _forward_eval(self, x, mask):
        enc = self.encoder
        xx = enc._check_input(x)
        eng = enc._ensure_engine()
        B, C, H, W = xx.shape
        N = enc._tokens(xx)
        pos = enc._mim_pos(xx)
        assert pos.shape[0] == N, "position table does not match the token count (img_size vs input size)"
        m = mask.detach().reshape(B, -1).to(device=xx.device, dtype=torch.float32).contiguous()
        x_rec = torch.empty_like(xx)
        sums = torch.empty(2, dtype=torch.float64, device=xx.device)
        chunk = max(1, min(enc.chunk_tiles, B))
        ws = enc._workspace(chunk, N, xx.device)
        check(_lib.load_library().vitocm_mim_forward(eng, ptr(xx), B, H, W, ptr(pos), ptr(m), ptr(x_rec), ptr(sums), ptr(ws),
                                                     ws.numel(), chunk, cur_stream()))
        loss = (sums[0] / (sums[1] + 1e-5) / self.in_chans).to(torch.float32)
        mask_up = mask.repeat_interleave(self.patch_size, 1).repeat_interleave(self.patch_size, 2).unsqueeze(1).contiguous()
        return loss, x_rec, mask_up

    @torch.jit.ignore
    def no_weight_decay(self):
        if hasattr(self.encoder, 'no_weight_decay'):
            return {'encoder.' + i for i in self.encoder.no_weight_decay()}
        return {}

    @torch.jit.ignore
    def no_weight_decay_keywords(self):
        if hasattr(self.encoder, 'no_weight_decay_keywords'):
            return {'encoder.' + i for i in self.encoder.no_weight_decay_keywords()}
        return {}


def build_model(args, depth=12, num_heads=6, precision="bf16"):
    """SSS/model.py:91-108.  The reference's build_model hard-codes depth=4 / num_heads=3 at embed_dim 384 (head_dim 128):
    ``build_model(args, depth=4, num_heads=3)`` builds exactly that encoder.  The defaults (12 blocks, 6 heads, head_dim 64)
    are the ViT-S/8 of the shipped training log (SSS/output/log_rank0.txt)."""
    return VisionTransformerForSimMIM(patch_size=args.MODEL.PATCH_SIZE, embed_dim=384, depth=depth, num_heads=num_heads,
                                      mlp_ratio=4, img_size=[args.DATA.IMG_SIZE], qkv_bias=True,
                                      norm_layer=partial(nn.LayerNorm, eps=1e-6), interpolate_encoding=True,
                                      precision=precision)
