"""Drop-in for the reference's ``dino.vision_transformer`` on B200.

Same constructor arguments, parameter names (state-dict keys) and methods as
Self-supervised_segmentation/dino/vision_transformer.py:135-279 of the reference
(``VisionTransformer``, ``vit_tiny`` / ``vit_small`` / ``vit_base``), but every forward runs in
libvitocm.so (hand-written sm_100a kernels behind a C ABI).  The torch modules below only own
the parameters -- they carry no arithmetic; there is no eager fallback.

Hot path: ``get_intermediate_feat(x, n=1)`` -> (feat, attns, qkvs) computes the last-layer CLS
attention rows eagerly with ``vitocm_forward_cls_attn`` and hands back *lazy* views for the
three lists; ``attns[0][0, :, 0, 1:]`` (the only slice the reference's callers read,
SSS/utils.py:232) is served from those rows, anything else materialises the full tensors
through the block-by-block entry points.
"""
from __future__ import annotations

import ctypes as C
import math
from functools import partial

import torch
import torch.nn as nn

from . import _lib
from ._lib import VitocmConfig, check, cur_stream, ptr

PRECISIONS = {"bf16": 0, "fp32": 1, "fp16": 2}


def parse_precision(spec: str, depth: int):
    """"bf16" | "fp32" | "fp16", optionally followed by "+mlp2" (every block) or "+mlp2:a-b,c" (blocks a..b and c): those blocks'
    fc1 / fc2 read their activations as (hi, lo) pairs (vitocm_set_layer_mode 1).  -> (engine precision, [mode per block])."""
    base, _, extra = spec.partition("+")
    if base not in PRECISIONS:
        raise ValueError(f"precision must start with one of {sorted(PRECISIONS)} (got {spec!r})")
    modes = [0] * depth
    if extra:
        kind, _, sel = extra.partition(":")
        if kind != "mlp2" or base == "fp32":
            raise ValueError(f"unknown precision schedule {spec!r} (bf16|fp16[+mlp2[:blocks]], fp32)")
        if not sel:
            modes = [1] * depth
        else:
            for part in sel.split(","):
                a, _, b = part.partition("-")
                for l in range(int(a), int(b or a) + 1):
                    if not 0 <= l < depth:
                        raise ValueError(f"block {l} out of range in {spec!r}")
                    modes[l] = 1
    return base, modes


def _trunc_normal_(t: torch.Tensor, std: float = 0.02, a: float = -2.0, b: float = 2.0) -> torch.Tensor:
    """Truncated-normal init with the reference's recipe (SSS/dino/utils.py:482-520)."""
    cdf = lambda v: (1.0 + math.erf(v / math.sqrt(2.0))) / 2.0   # noqa: E731
    lo, hi = cdf(a / std), cdf(b / std)
    with torch.no_grad():
        t.uniform_(2 * lo - 1, 2 * hi - 1).erfinv_().mul_(std * math.sqrt(2.0)).clamp_(min=a, max=b)
    return t


# --------------------------------------------------------------------------- parameter containers
class _Mlp(nn.Module):
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.fc2 = nn.Linear(hidden, dim)


class _Attention(nn.Module):
    def __init__(self, dim, num_heads, qkv_bias):
        super().__init__()
        self.num_heads = num_heads
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.proj = nn.Linear(dim, dim)


class _Block(nn.Module):
    def __init__(self, dim, num_heads, mlp_ratio, qkv_bias, norm_layer):
        super().__init__()
        self.norm1 = norm_layer(dim)
        self.attn = _Attention(dim, num_heads, qkv_bias)
        self.norm2 = norm_layer(dim)
        self.mlp = _Mlp(dim, int(dim * mlp_ratio))


class _PatchEmbed(nn.Module):
    def __init__(self, img_size, patch_size, in_chans, embed_dim):
        super().__init__()
        self.img_size = img_size
        self.patch_size = patch_size
        self.num_patches = (img_size // patch_size) ** 2
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size)


# --------------------------------------------------------------------------- lazy results
class LazyTensor:
    """A tensor computed on first use.  Quacks like the tensor it stands for."""

    def __init__(self, shape, producer):
        self._shape = torch.Size(shape)
        self._producer = producer
        self._value = None

    def materialize(self) -> torch.Tensor:
        if self._value is None:
            self._value = self._producer()
            assert tuple(self._value.shape) == tuple(self._shape), (self._value.shape, self._shape)
        return self._value

    @property
    def shape(self):
        return self._shape

    def size(self, dim=None):
        return self._shape if dim is None else self._shape[dim]

    def dim(self):
        return len(self._shape)

    def __len__(self):
        return self._shape[0]

    def __getitem__(self, idx):
        return self.materialize()[idx]

    def __getattr__(self, name):          # anything else: behave as the real tensor
        if name.startswith("_"):
            raise AttributeError(name)
        return getattr(self.materialize(), name)

    @classmethod
    def __torch_function__(cls, func, types, args=(), kwargs=None):
        kwargs = kwargs or {}
        unwrap = lambda a: a.materialize() if isinstance(a, LazyTensor) else a   # noqa: E731
        return func(*[unwrap(a) for a in args], **{k: unwrap(v) for k, v in kwargs.items()})


class LazyAttention(LazyTensor):
    """``attn`` of a block, [B, heads, N, N].  ``attn[b, :, 0, c]`` (CLS query, any column index)
    is answered from the eagerly computed CLS rows; everything else materialises N x N."""

    def __init__(self, shape, producer, cls_rows: torch.Tensor, row_fn=None):
        super().__init__(shape, producer)
        self.cls_rows = cls_rows                    # [B, heads, N] fp32, device
        self._row_fn = row_fn                       # q -> [B, heads, N] rows of query token q (computed on demand)
        self._rows = {0: cls_rows}

    def __getitem__(self, idx):
        if self._value is None and isinstance(idx, tuple) and len(idx) >= 3:
            q = idx[2]
            if isinstance(q, int):
                q = q % self._shape[2]
                if q not in self._rows and self._row_fn is not None:
                    self._rows[q] = self._row_fn(q)      # region query (SSS/analyse_attention.py:183-247) without N x N
                if q in self._rows:
                    return self._rows[q][(idx[0], idx[1]) + tuple(idx[3:])]
        return self.materialize()[idx]


# --------------------------------------------------------------------------- the model
class VisionTransformer(nn.Module):
    """Vision Transformer whose forward passes run in libvitocm (B200 / sm_100a).

    Constructor signature follows the reference (vit.py:137-139); ``precision`` ("bf16" |
    "fp16" | "fp32", see parse_precision), ``chunk_tiles`` (tiles per kernel launch) and ``lanes`` (chunks in flight on concurrent streams) are additions.  Dropout / stochastic depth must be 0 (the
    reference's inference and MIM configurations all use 0)."""

    def __init__(self, img_size=[224], patch_size=16, in_chans=3, num_classes=0, embed_dim=768, depth=12,
                 num_heads=12, mlp_ratio=4., qkv_bias=False, qk_scale=None, drop_rate=0., attn_drop_rate=0.,
                 drop_path_rate=0., norm_layer=nn.LayerNorm, precision="bf16", chunk_tiles=512, lanes=1, **kwargs):
        super().__init__()
        if drop_rate or attn_drop_rate or drop_path_rate:
            raise NotImplementedError("vitocm: dropout / drop-path rates must be 0 on this path")
        if embed_dim % num_heads or embed_dim // num_heads not in (64, 128):
            raise NotImplementedError("vitocm kernels support head_dim 64 and 128 (embed_dim %d / num_heads %d)"
                                      % (embed_dim, num_heads))
        parse_precision(precision, depth)
        self.num_features = self.embed_dim = embed_dim
        self.num_heads = num_heads
        self.depth = depth
        self.mlp_ratio = mlp_ratio
        self.in_chans = in_chans
        self.precision = precision
        self.chunk_tiles = chunk_tiles
        self.lanes = int(lanes)          # chunks processed concurrently by cls_attention_rows (vitocm_set_concurrency)
        self.qk_scale = qk_scale or (embed_dim // num_heads) ** -0.5

        self.patch_embed = _PatchEmbed(img_size[0], patch_size, in_chans, embed_dim)
        n = self.patch_embed.num_patches
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, n + 1, embed_dim))
        self.blocks = nn.ModuleList([_Block(embed_dim, num_heads, mlp_ratio, qkv_bias, norm_layer) for _ in range(depth)])
        self.norm = norm_layer(embed_dim)
        self.head = nn.Linear(embed_dim, num_classes) if num_classes > 0 else nn.Identity()
        self.ln_eps = float(self.norm.eps)

        _trunc_normal_(self.pos_embed, std=.02)
        _trunc_normal_(self.cls_token, std=.02)
        for m in self.modules():                   # vit.py:166-174
            if isinstance(m, nn.Linear):
                _trunc_normal_(m.weight, std=.02)
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.LayerNorm):
                nn.init.constant_(m.bias, 0)
                nn.init.constant_(m.weight, 1.0)

        self._engine = None
        self._engine_key = None
        self._pos_cache = {}
        self._ws = None
        # a buffer so that it follows .cuda() and the engine can bind it in place like the parameters (training)
        self.register_buffer("_zero_qkv_bias", torch.zeros(3 * embed_dim), persistent=False)
        self._train_ws = None          # the differentiable forward's saved activations (vitocm_encoder_train_forward)
        self._train_ws_gen = 0
        self._grads_bound_to = None    # MIM's gradient buffers when they are the ones bound (vitocm_bind_grad); None otherwise

    # ------------------------------------------------------------------ engine plumbing
    def _engine_params(self):
        """(state-dict key, tensor) for everything the C engine needs."""
        out = [("cls_token", self.cls_token), ("patch_embed.proj.weight", self.patch_embed.proj.weight),
               ("patch_embed.proj.bias", self.patch_embed.proj.bias), ("norm.weight", self.norm.weight),
               ("norm.bias", self.norm.bias)]
        if hasattr(self, "mask_token"):
            out.append(("mask_token", self.mask_token))
        extra = getattr(self, "_extra_engine_params", None)     # e.g. the MIM decoder (model.py)
        if extra is not None:
            out += list(extra())
        for i, blk in enumerate(self.blocks):
            pre = f"blocks.{i}."
            qkv_b = blk.attn.qkv.bias if blk.attn.qkv.bias is not None else self._zero_qkv_bias
            out += [(pre + "norm1.weight", blk.norm1.weight), (pre + "norm1.bias", blk.norm1.bias),
                    (pre + "attn.qkv.weight", blk.attn.qkv.weight), (pre + "attn.qkv.bias", qkv_b),
                    (pre + "attn.proj.weight", blk.attn.proj.weight), (pre + "attn.proj.bias", blk.attn.proj.bias),
                    (pre + "norm2.weight", blk.norm2.weight), (pre + "norm2.bias", blk.norm2.bias),
                    (pre + "mlp.fc1.weight", blk.mlp.fc1.weight), (pre + "mlp.fc1.bias", blk.mlp.fc1.bias),
                    (pre + "mlp.fc2.weight", blk.mlp.fc2.weight), (pre + "mlp.fc2.bias", blk.mlp.fc2.bias)]
        return out

    def _weights_key(self):
        return (self.precision, torch.cuda.current_device(),
                tuple((p.data_ptr(), p._version) for _, p in self._engine_params()), self.pos_embed._version)

    def _bindable(self):
        """Training mode: every engine parameter is fp32, contiguous, 16-byte aligned and already on the current
        device, so the engine can use the storage in place (vitocm_bind_weight) instead of a host round trip."""
        dev = torch.cuda.current_device()
        return all(p.is_cuda and p.device.index == dev and p.dtype == torch.float32 and p.is_contiguous() and p.data_ptr() % 16 == 0
                   for _, p in self._engine_params())

    def refresh_engine(self):
        """(Re)load the parameters into the C engine: repack to bf16 hi/lo etc.  With ``self._bind_weights`` set (the
        training path) the engine aliases the parameters' device storage and a change of their values only costs an
        asynchronous repack (vitocm_refresh_weights)."""
        lib = _lib.load_library()
        if not torch.cuda.is_available():
            raise _lib.VitocmError("vitocm needs a CUDA device (B200, sm_100a); there is no CPU path")
        if self._engine is None:
            base, modes = parse_precision(self.precision, self.depth)
            cfg = VitocmConfig(self.embed_dim, self.depth, self.num_heads, int(self.embed_dim * self.mlp_ratio),
                               self.patch_embed.patch_size, self.in_chans, self.ln_eps, float(self.qk_scale),
                               PRECISIONS[base])
            handle = C.c_void_p()
            check(lib.vitocm_create(C.byref(cfg), C.byref(handle)))
            for l, m in enumerate(modes):
                if m:
                    check(lib.vitocm_set_layer_mode(handle, l, m))
            self._engine = handle
            self._bound_ptrs = None
            check(lib.vitocm_set_concurrency(handle, self.lanes))
        if getattr(self, "_bind_weights", False) and self._bindable():
            ptrs = tuple(p.data_ptr() for _, p in self._engine_params())
            if ptrs != self._bound_ptrs:
                for name, p in self._engine_params():
                    check(lib.vitocm_bind_weight(self._engine, name.encode(), p.data_ptr(), p.numel()))
                check(lib.vitocm_finalize_weights(self._engine))
                self._bound_ptrs = ptrs
            else:
                check(lib.vitocm_refresh_weights(self._engine, cur_stream()))
        else:
            for name, p in self._engine_params():
                host = p.detach().to(device="cpu", dtype=torch.float32).contiguous()
                check(lib.vitocm_load_weight(self._engine, name.encode(), host.data_ptr(), host.numel()))
            check(lib.vitocm_finalize_weights(self._engine))
            self._bound_ptrs = None
        self._engine_key = self._weights_key()
        self._pos_cache = {}

    def _ensure_engine(self):
        if self._engine is None or self._engine_key != self._weights_key():
            self.refresh_engine()
        return self._engine

    def __del__(self):
        eng = getattr(self, "_engine", None)
        if eng is not None and _lib._lib is not None:
            try:
                _lib._lib.vitocm_destroy(eng)
            except Exception:
                pass

    def set_precision(self, precision: str):
        parse_precision(precision, self.depth)
        if precision != self.precision:
            self.precision = precision
            if self._engine is not None:
                _lib.load_library().vitocm_destroy(self._engine)
                self._engine = None
        return self

    def _workspace(self, tiles: int, n_tokens: int, device) -> torch.Tensor:
        need = int(_lib.load_library().vitocm_workspace_bytes(self._engine, tiles, n_tokens))
        if self._ws is None or self._ws.numel() < need or self._ws.device != device:
            self._ws = torch.empty(need, dtype=torch.uint8, device=device)
        return self._ws

    # ------------------------------------------------------------------ position table
    def interpolate_pos_encoding(self, x, w, h):
        """vit.py:176-196.  `x` only supplies the token count, as in the reference."""
        npatch = x.shape[1] - 1
        return self._pos_table(npatch, w, h).unsqueeze(0)

    def _pos_table(self, npatch: int, w: int, h: int) -> torch.Tensor:
        """[1 + npatch, D] fp32 on the current device; bicubic resize of the stored table when the
        input is not the constructor size (frozen weights -> computed once per shape and cached)."""
        dev = torch.device("cuda", torch.cuda.current_device())
        key = (npatch, w, h, dev)
        hit = self._pos_cache.get(key)
        if hit is not None:
            return hit
        table = self._pos_graph(npatch, w, h, self.pos_embed.detach().to(device=dev, dtype=torch.float32)).contiguous()
        self._pos_cache[key] = table
        return table

    def _pos_graph(self, npatch: int, w: int, h: int, pos=None) -> torch.Tensor:
        """vit.py:176-196 as torch operations on ``pos`` (default: ``pos_embed`` itself, so that the table is differentiable
        with respect to it) -> [1 + npatch, D].  ``w``, ``h``: the input's dims 2 and 3, named as in the reference."""
        pos = self.pos_embed if pos is None else pos
        N = pos.shape[1] - 1
        if not (npatch == N and w == h):
            p = self.patch_embed.patch_size
            dim = pos.shape[-1]
            w0, h0 = w // p + 0.1, h // p + 0.1
            s = int(math.sqrt(N))
            grid = nn.functional.interpolate(pos[:, 1:].reshape(1, s, s, dim).permute(0, 3, 1, 2),
                                             scale_factor=(w0 / math.sqrt(N), h0 / math.sqrt(N)), mode="bicubic")
            assert int(w0) == grid.shape[-2] and int(h0) == grid.shape[-1]
            pos = torch.cat((pos[:, :1], grid.permute(0, 2, 3, 1).reshape(1, -1, dim)), dim=1)
        return pos[0]

    # ------------------------------------------------------------------ C-ABI calls
    def _check_input(self, x, allow_gray: bool = False):
        if x.dim() != 4 or (x.shape[1] != self.in_chans and not (allow_gray and x.shape[1] == 1)):
            raise ValueError(f"expected [B,{self.in_chans},H,W], got {tuple(x.shape)}")
        p = self.patch_embed.patch_size
        if x.shape[2] % p or x.shape[3] % p:
            raise ValueError("H and W must be multiples of the patch size")
        if not x.is_cuda:
            raise _lib.VitocmError("vitocm: input must be a CUDA tensor (no CPU path)")
        return x.detach().to(torch.float32).contiguous()

    def _tokens(self, x):
        p = self.patch_embed.patch_size
        return (x.shape[2] // p) * (x.shape[3] // p) + 1

    @torch.no_grad()
    def cls_attention_rows(self, x: torch.Tensor) -> torch.Tensor:
        """get_last_selfattention(x)[:, :, 0, :] -> [B, heads, N] fp32, without forming N x N.

        A single-channel ``x`` [B, 1, H, W] on a multi-channel model is the gray fast path: it stands for the image with all
        channels equal (what the reference feeds for every OCM tile) and runs the channel-folded patch filter."""
        x = self._check_input(x, allow_gray=True)
        eng = self._ensure_engine()
        B, Cx, H, W = x.shape
        N = self._tokens(x)
        pos = self._pos_table(N - 1, H, W)
        chunk = max(1, min(self.chunk_tiles, B))
        ws = self._workspace(chunk, N, x.device)
        out = torch.empty(B, self.num_heads, N, dtype=torch.float32, device=x.device)
        fn = _lib.load_library().vitocm_forward_cls_attn_gray if (Cx == 1 and self.in_chans > 1) else _lib.load_library().vitocm_forward_cls_attn
        check(fn(eng, ptr(x), B, H, W, ptr(pos), ptr(out), ptr(ws), ws.numel(), chunk, cur_stream()))
        return out

    @torch.no_grad()
    def cls_attention_rows_mosaic(self, mosaic: torch.Tensor, grid, window: int, stride: int, t0: int, count: int) -> torch.Tensor:
        """cls_attention_rows of the windows t0 .. t0+count-1 (row-major in the sliding-window grid, SSS/sw_processing.py:151-163)
        of a gray uint8 CUDA mosaic, cut out by the patch-embedding producer itself: no crop is ever materialised.  grid: n for an
        n x n grid, or (ny, nx) for a rectangular one (ny rows of windows over the height, nx columns over the width; window t
        has origin ((t // nx) * stride, (t % nx) * stride)).  -> [count, heads, N] fp32."""
        ny, nx = (grid, grid) if isinstance(grid, int) else (int(grid[0]), int(grid[1]))
        if isinstance(mosaic, tuple):      # (device address of row 0, height, width, pitch, device): a band buffer addressed by absolute rows
            mos_ptr, mos_h, mos_w, pitch, dev = mosaic
        else:
            if mosaic.dtype != torch.uint8 or mosaic.dim() != 2 or not mosaic.is_cuda or mosaic.stride(1) != 1:
                raise ValueError("mosaic must be a 2-D uint8 CUDA tensor with unit column stride")
            mos_ptr, mos_h, mos_w, pitch, dev = mosaic.data_ptr(), mosaic.shape[0], mosaic.shape[1], mosaic.stride(0), mosaic.device
        if self.in_chans < 2:
            raise NotImplementedError("mosaic ingest runs the channel-folded (gray) patch filter of a multi-channel model")
        p = self.patch_embed.patch_size
        if window % p:
            raise ValueError("window must be a multiple of the patch size")
        eng = self._ensure_engine()
        N = (window // p) ** 2 + 1
        pos = self._pos_table(N - 1, window, window)
        chunk = max(1, min(self.chunk_tiles, count))
        ws = self._workspace(chunk, N, dev)
        out = torch.empty(count, self.num_heads, N, dtype=torch.float32, device=dev)
        check(_lib.load_library().vitocm_forward_cls_attn_mosaic_grid(eng, mos_ptr, mos_h, mos_w, pitch, ny, nx,
                                                                      window, stride, t0, count, ptr(pos), ptr(out), ptr(ws), ws.numel(), chunk,
                                                                      cur_stream()))
        return out

    @torch.no_grad()
    def attention_rows(self, x: torch.Tensor, queries, return_keys: bool = False):
        """get_last_selfattention(x)[:, :, queries, :] -> [B, heads, nq, N] fp32 for a list of query tokens (0 = CLS,
        1 + i = patch i; SSS/analyse_attention.py:183-247 region queries), without forming N x N.  With ``return_keys``
        also the last block's K features [B, heads, N, head_dim] (= qkv[1] of get_intermediate_feat; SSS/eval.py:186-202)."""
        x = self._check_input(x)
        eng = self._ensure_engine()
        B, _, H, W = x.shape
        N = self._tokens(x)
        q = torch.as_tensor(queries, dtype=torch.int32).reshape(-1)
        if q.numel() == 0 or int(q.min()) < -N or int(q.max()) >= N:
            raise IndexError(f"query tokens must lie in [0, {N})")
        q = (q % N).to(device=x.device).contiguous()
        pos = self._pos_table(N - 1, H, W)
        chunk = max(1, min(self.chunk_tiles, B))
        ws = self._workspace(chunk, N, x.device)
        out = torch.empty(B, self.num_heads, q.numel(), N, dtype=torch.float32, device=x.device)
        keys = torch.empty(B, N, self.embed_dim, dtype=torch.float32, device=x.device) if return_keys else None
        check(_lib.load_library().vitocm_forward_query_attn(eng, ptr(x), B, H, W, ptr(pos), ptr(q), q.numel(), ptr(out), ptr(keys), ptr(ws),
                                                            ws.numel(), chunk, cur_stream()))
        if return_keys:
            return out, keys.reshape(B, N, self.num_heads, self.embed_dim // self.num_heads).permute(0, 2, 1, 3)
        return out

    @torch.no_grad()
    def prepare_tokens(self, x, mask=None):
        """vit.py:198-209 -> [B, N, D] fp32."""
        x = self._check_input(x)
        eng = self._ensure_engine()
        B, _, H, W = x.shape
        N = self._tokens(x)
        pos = self._pos_table(N - 1, H, W)
        X = torch.empty(B, N, self.embed_dim, dtype=torch.float32, device=x.device)
        m = None if mask is None else mask.detach().reshape(B, -1).to(device=x.device, dtype=torch.float32).contiguous()
        check(_lib.load_library().vitocm_prepare_tokens(eng, ptr(x), B, H, W, ptr(pos), ptr(m), ptr(X), cur_stream()))
        return X

    def _run_blocks(self, X, first, last):
        """Blocks [first, last) in place on X [B, N, D], chunked over the batch."""
        lib = _lib.load_library()
        B, N, _ = X.shape
        chunk = max(1, min(self.chunk_tiles, B))
        ws = self._workspace(chunk, N, X.device)
        for b0 in range(0, B, chunk):
            xb = X[b0:b0 + chunk]
            for layer in range(first, last):
                check(lib.vitocm_block_forward(self._engine, layer, ptr(xb), xb.shape[0], N, ptr(ws), ws.numel(), cur_stream()))
        return X

    def _attn_probs(self, X, layer):
        lib = _lib.load_library()
        B, N, D = X.shape
        attn = torch.empty(B, self.num_heads, N, N, dtype=torch.float32, device=X.device)
        qkv = torch.empty(B * N, 3 * D, dtype=torch.float32, device=X.device)
        chunk = max(1, min(self.chunk_tiles, B))
        ws = self._workspace(chunk, N, X.device)
        for b0 in range(0, B, chunk):
            xb, ab, qb = X[b0:b0 + chunk], attn[b0:b0 + chunk], qkv[b0 * N:(b0 + chunk) * N]
            check(lib.vitocm_block_attn_probs(self._engine, layer, ptr(xb), xb.shape[0], N, ptr(ab), ptr(qb), ptr(ws),
                                              ws.numel(), cur_stream()))
        # [B*N, 3D] -> [3, B, heads, N, dh]  (vit.py:80 reshape/permute; a view, no arithmetic)
        qkv = qkv.reshape(B, N, 3, self.num_heads, D // self.num_heads).permute(2, 0, 3, 1, 4)
        return attn, qkv

    def _final_norm(self, X):
        B, N, D = X.shape
        out = torch.empty_like(X)
        check(_lib.load_library().vitocm_final_norm(self._engine, ptr(X), ptr(out), B * N, cur_stream()))
        return out

    # ------------------------------------------------------------------ training (fine-tuning, linear probing)
    def _differentiable(self, x) -> bool:
        """The gate of forward_feats / forward / get_intermediate_layers: with gradients enabled, a call is differentiable
        when ``x`` requires grad or, in training mode, when an engine parameter does (MIM.forward's rule).  Every other call
        (no_grad, eval(), frozen parameters) runs the inference path."""
        if not torch.is_grad_enabled():
            return False
        if isinstance(x, torch.Tensor) and x.requires_grad:
            return True
        return self.training and (self.pos_embed.requires_grad or any(p.requires_grad for p in self._encoder_grad_params().values()))

    def _encoder_grad_params(self):
        """{engine name: parameter} of everything vitocm_encoder_backward writes a gradient for (pos_embed excepted: its gradient
        is dpos, carried through the position-table graph).  A qkv bias that does not exist gets none."""
        return {n: p for n, p in self._engine_params() if n != "mask_token" and not n.startswith("decoder.") and p is not self._zero_qkv_bias}

    def _encoder_train(self, x, n_out: int):
        """Differentiable [norm(x_l) for the last n_out blocks] through vitocm_encoder_train_forward / vitocm_encoder_backward."""
        if parse_precision(self.precision, self.depth)[0] == "fp32":
            raise _lib.VitocmError("vitocm: training runs on bf16 or fp16 engines only; build the encoder with precision='bf16' or "
                                   "'fp16' (or call it under torch.no_grad() / .eval() for fp32-parity inference)")
        if x.dim() == 4 and x.shape[1] == 1 and self.in_chans > 1:
            raise _lib.VitocmError(f"vitocm: gray [B, 1, H, W] inputs have no backward; pass the {self.in_chans}-channel image, "
                                   f"e.g. x.expand(-1, {self.in_chans}, -1, -1), or call under torch.no_grad()")
        n_out = min(n_out, self.depth)            # as the reference: n > depth gives every block, n < 1 none
        if n_out < 1:
            return []
        xx = self._check_input(x)
        self._bind_weights = True                 # the optimizer updates the parameters in place: repack on the device
        self._ensure_engine()
        _, _, H, W = xx.shape
        N = self._tokens(xx)
        pos = self._pos_graph(N - 1, H, W)
        named = self._encoder_grad_params()
        feats = _EncoderStep.apply(self, x, xx, n_out, pos, tuple(named), *named.values())
        return list(feats.unbind(0))

    def _bind_encoder_grads(self, names, dev):
        """A fresh zeroed flat fp32 buffer for one backward's parameter gradients (returned to autograd as views, so .grad may
        keep them), bound to the engine for that backward only (see _unbind_encoder_grads).  Slots are 16-byte aligned; a missing
        qkv bias accumulates into a scratch slot.  -> ({name: view} for ``names``, every bound name)."""
        eng = self._engine
        sizes = {n: p.numel() for n, p in self._engine_params() if n != "mask_token" and not n.startswith("decoder.")}
        offs, total = {}, 0
        for n, k in sizes.items():
            offs[n] = total
            total += (k + 3) // 4 * 4
        flat = torch.zeros(total, dtype=torch.float32, device=dev)
        lib = _lib.load_library()
        self._grads_bound_to = None         # the next MIM backward rebinds its own buffers
        for n, o in offs.items():
            check(lib.vitocm_bind_grad(eng, n.encode(), flat.data_ptr() + 4 * o))
        return {n: flat[offs[n]:offs[n] + sizes[n]] for n in names}, list(offs)

    def _unbind_encoder_grads(self, bound):
        """After the backward's launches: the engine must not keep addresses into a buffer that autograd may free (a later
        backward that does not bind a name, e.g. MIM's with no qkv bias, then fails with 'no bound gradient buffer')."""
        lib = _lib.load_library()
        for n in bound:
            check(lib.vitocm_bind_grad(self._engine, n.encode(), None))

    # ------------------------------------------------------------------ reference methods
    def forward_feats(self, x):
        """vit.py:218-223 -> norm(x) [B, N, D]; differentiable under the rule of ``_differentiable``."""
        if self._differentiable(x):
            return self._encoder_train(x, 1)[0]
        return self._forward_feats(x)

    @torch.no_grad()
    def _forward_feats(self, x):
        X = self.prepare_tokens(x)
        self._run_blocks(X, 0, self.depth)
        return self._final_norm(X)

    def forward(self, x):
        """vit.py:211-216 -> CLS embedding [B, D]."""
        return self.forward_feats(x)[:, 0]

    @torch.no_grad()
    def get_last_selfattention(self, x):
        """vit.py:239-246 -> attention of the last block, [B, heads, N, N] fp32."""
        X = self.prepare_tokens(x)
        self._run_blocks(X, 0, self.depth - 1)
        return self._attn_probs(X, self.depth - 1)[0]

    def get_intermediate_layers(self, x, n=1):
        """vit.py:248-256 -> [norm(x_i)] for the n last blocks; differentiable under the rule of ``_differentiable``."""
        if self._differentiable(x):
            return self._encoder_train(x, n)
        return self._get_intermediate_layers(x, n)

    @torch.no_grad()
    def _get_intermediate_layers(self, x, n):
        X = self.prepare_tokens(x)
        outs = []
        for i in range(self.depth):
            self._run_blocks(X, i, i + 1)
            if self.depth - i <= n:
                outs.append(self._final_norm(X))
        return outs

    @torch.no_grad()
    def _intermediate_full(self, x, n):
        X = self.prepare_tokens(x)
        feat, attns, qkvs = [], [], []
        for i in range(self.depth):
            if self.depth - i <= n:
                a, q = self._attn_probs(X, i)
                attns.append(a)
                qkvs.append(q)
            self._run_blocks(X, i, i + 1)
            if self.depth - i <= n:
                feat.append(self._final_norm(X))
        return feat, attns, qkvs

    @torch.no_grad()
    def get_intermediate_feat(self, x, n=1, lazy=True):
        """vit.py:225-237 -> (feat list, attn list, qkv list) for the n last blocks.

        With ``lazy`` (default) and n == 1 only the CLS attention rows are computed now; the
        returned objects materialise the full tensors on demand (see module docstring)."""
        if not lazy or n != 1:
            return self._intermediate_full(x, n)
        rows = self.cls_attention_rows(x)
        B, H, N = rows.shape
        D = self.embed_dim
        cache = {}

        def full():
            if "v" not in cache:
                cache["v"] = self._intermediate_full(x, 1)
            return cache["v"]

        feat = LazyTensor((B, N, D), lambda: full()[0][0])
        attn = LazyAttention((B, H, N, N), lambda: full()[1][0], rows, row_fn=lambda q: self.attention_rows(x, [q])[:, :, 0, :])
        qkv = LazyTensor((3, B, H, N, D // H), lambda: full()[2][0])
        return [feat], [attn], [qkv]


class _EncoderStep(torch.autograd.Function):
    """feats [n_out, B, N, D] = norm(x_l) of the last n_out blocks, with vitocm_encoder_backward as the backward.  The parameters
    are inputs, and their gradients come back through autograd, so .grad accumulation, hooks, optimizers and
    torch.autograd.grad work as for any module.  ``x`` is an input for dx; ``xx`` is its fp32 contiguous copy the kernels read."""

    @staticmethod
    def forward(ctx, enc, x, xx, n_out, pos, names, *params):
        lib = _lib.load_library()
        eng = enc._engine
        B, _, H, W = xx.shape
        N = enc._tokens(xx)
        need = int(lib.vitocm_mim_train_workspace_bytes(eng, B, N))
        if enc._train_ws is None or enc._train_ws.numel() < need or enc._train_ws.device != xx.device:
            enc._train_ws = None
            enc._train_ws = torch.empty(need, dtype=torch.uint8, device=xx.device)
        posc = pos.detach().to(torch.float32).contiguous()
        feats = torch.empty(n_out, B, N, enc.embed_dim, dtype=torch.float32, device=xx.device)
        check(lib.vitocm_encoder_train_forward(eng, ptr(xx), B, H, W, ptr(posc), n_out, ptr(feats), ptr(enc._train_ws),
                                               enc._train_ws.numel(), cur_stream()))
        # the saved activations live in the encoder's one training workspace: stamp it, so that a backward whose forward has since
        # been overwritten by another differentiable forward fails loudly instead of producing wrong gradients
        enc._train_ws_gen += 1
        ctx.enc, ctx.ws_gen, ctx.n_out, ctx.names = enc, enc._train_ws_gen, n_out, names
        ctx.pos_shape, ctx.x_dtype, ctx.shapes = tuple(pos.shape), x.dtype, [p.shape for p in params]
        ctx.save_for_backward(xx)
        return feats

    @staticmethod
    def backward(ctx, dfeats):
        enc = ctx.enc
        if torch.is_grad_enabled():
            raise _lib.VitocmError("vitocm: the encoder's backward is not differentiable (double backward); "
                                   "call backward() / torch.autograd.grad without create_graph=True")
        if ctx.ws_gen != enc._train_ws_gen:
            raise _lib.VitocmError("vitocm: the activations of this forward were overwritten by a later differentiable forward "
                                   "(call backward() before the next forward, or run evaluation under torch.no_grad() / .eval())")
        xx, = ctx.saved_tensors
        B, C, H, W = xx.shape
        dpos = torch.empty(ctx.pos_shape, dtype=torch.float32, device=xx.device)
        dx = torch.empty_like(xx) if ctx.needs_input_grad[1] else None
        dfe = dfeats.detach().to(torch.float32).contiguous()
        grads, bound = enc._bind_encoder_grads(ctx.names, xx.device)
        try:
            check(_lib.load_library().vitocm_encoder_backward(enc._engine, ptr(xx), B, H, W, ctx.n_out, ptr(dfe), ptr(dpos), ptr(dx),
                                                              ptr(enc._train_ws), enc._train_ws.numel(), cur_stream()))
        finally:
            enc._unbind_encoder_grads(bound)
        param_grads = [grads[n].view(shape) for n, shape in zip(ctx.names, ctx.shapes)]
        return (None, None if dx is None else dx.to(ctx.x_dtype), None, None, dpos, None, *param_grads)


def vit_tiny(patch_size=16, **kwargs):
    return VisionTransformer(patch_size=patch_size, embed_dim=192, depth=12, num_heads=3, mlp_ratio=4, qkv_bias=True,
                             norm_layer=partial(nn.LayerNorm, eps=1e-6), **kwargs)


def vit_small(patch_size=16, **kwargs):
    return VisionTransformer(patch_size=patch_size, embed_dim=384, depth=12, num_heads=6, mlp_ratio=4, qkv_bias=True,
                             norm_layer=partial(nn.LayerNorm, eps=1e-6), **kwargs)


def vit_base(patch_size=16, **kwargs):
    return VisionTransformer(patch_size=patch_size, embed_dim=768, depth=12, num_heads=12, mlp_ratio=4, qkv_bias=True,
                             norm_layer=partial(nn.LayerNorm, eps=1e-6), **kwargs)
