"""ctypes binding of libvitocm.so (include/vitocm.h).  There is no CPU or eager-PyTorch fallback:
if the CUDA library is missing or a call fails, this module raises."""
from __future__ import annotations

import ctypes as C
import os

import torch

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# VITOCM_LIB: another build of the same library (A/B timing of two builds on one box); the default is the in-tree one
LIB_PATH = os.environ.get("VITOCM_LIB") or os.path.join(PKG_DIR, "libvitocm.so")

c_void_p, c_int, c_int64, c_size_t, c_float, c_char_p = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_float, C.c_char_p


class VitocmConfig(C.Structure):
    _fields_ = [("embed_dim", c_int), ("depth", c_int), ("num_heads", c_int), ("mlp_hidden", c_int),
                ("patch_size", c_int), ("in_chans", c_int), ("ln_eps", c_float), ("qk_scale", c_float),
                ("precision", c_int)]


# name -> (restype, argtypes); mirrors include/vitocm.h one to one
SIGNATURES = {
    "vitocm_version": (c_int, []),
    "vitocm_last_error": (c_char_p, []),
    "vitocm_create": (c_int, [C.POINTER(VitocmConfig), C.POINTER(c_void_p)]),
    "vitocm_destroy": (c_int, [c_void_p]),
    "vitocm_load_weight": (c_int, [c_void_p, c_char_p, c_void_p, c_int64]),
    "vitocm_finalize_weights": (c_int, [c_void_p]),
    "vitocm_workspace_bytes": (c_size_t, [c_void_p, c_int, c_int]),
    "vitocm_set_concurrency": (c_int, [c_void_p, c_int]),
    "vitocm_set_layer_mode": (c_int, [c_void_p, c_int, c_int]),
    "vitocm_forward_cls_attn": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
                                        c_int, c_void_p]),
    "vitocm_forward_cls_attn_gray": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
                                             c_int, c_void_p]),
    "vitocm_forward_cls_attn_mosaic": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                               c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "vitocm_forward_cls_attn_mosaic_grid": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_int, c_int, c_int, c_int, c_int,
                                                    c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "vitocm_forward_query_attn": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                          c_size_t, c_int, c_void_p]),
    "vitocm_prepare_tokens": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vitocm_block_forward": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "vitocm_block_attn_probs": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
                                        c_void_p]),
    "vitocm_mim_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                   c_int, c_void_p]),
    "vitocm_final_norm": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "vitocm_head_mean": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "vitocm_attn_cummass": (c_int, [c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "vitocm_tile_threshold": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_void_p]),
    "vitocm_extract_tiles": (c_int, [c_void_p, c_int, c_int, c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                     c_void_p]),
    "vitocm_tile_threshold_aux": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_void_p, c_void_p, c_void_p]),
    "vitocm_stitch_result": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                     c_void_p, c_void_p, c_void_p, c_void_p]),
    "vitocm_stitch_gray": (c_int, [c_void_p, c_int, c_int, c_int64, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p,
                                   c_void_p]),
    "vitocm_minmax_init": (c_int, [c_void_p, c_void_p]),
    "vitocm_stitch_minmax": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p,
                                     c_void_p, c_void_p, c_void_p]),
    "vitocm_stitch_hist": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                   c_void_p, c_void_p, c_void_p]),
    "vitocm_otsu": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "vitocm_stitch_mask": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vitocm_concat_crops_f32": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "vitocm_concat_crops_u8": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "vitocm_extract_tiles_grid": (c_int, [c_void_p, c_int, c_int, c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                          c_void_p]),
    "vitocm_stitch_gray_grid": (c_int, [c_void_p, c_int, c_int, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p,
                                        c_void_p]),
    "vitocm_stitch_minmax_grid": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p,
                                          c_void_p, c_void_p, c_void_p]),
    "vitocm_stitch_hist_grid": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                        c_void_p, c_void_p, c_void_p]),
    "vitocm_stitch_mask_grid": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vitocm_stitch_result_grid": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                          c_void_p, c_void_p, c_void_p, c_void_p]),
    "vitocm_concat_crops_grid_f32": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "vitocm_concat_crops_grid_u8": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "vitocm_concat_crops_overlap_f32": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "vitocm_concat_crops_overlap_u8": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "vitocm_concat_grid_f32": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "vitocm_crop_u8": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "vitocm_gemm": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p,
                            c_void_p, c_int64, c_int, c_int, c_void_p]),
    "vitocm_gemm_ln": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_int64, c_void_p]),
    "vitocm_mlp_fused": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_void_p,
                                 c_void_p, c_void_p]),
    "vitocm_mlp_fused_timeline": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_int, c_void_p,
                                          c_void_p, c_void_p, c_void_p, c_void_p]),
    "vitocm_block_tail": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64,
                                  c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                                  c_void_p, c_int64, c_void_p, c_void_p]),
    "vitocm_attention": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_int64, c_void_p]),
    "vitocm_attention_timeline": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    "vitocm_layernorm": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_void_p]),
    "vitocm_bind_weight": (c_int, [c_void_p, c_char_p, c_void_p, c_int64]),
    "vitocm_refresh_weights": (c_int, [c_void_p, c_void_p]),
    "vitocm_bind_grad": (c_int, [c_void_p, c_char_p, c_void_p]),
    "vitocm_mim_train_workspace_bytes": (c_size_t, [c_void_p, c_int, c_int]),
    "vitocm_mim_train_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_size_t, c_void_p]),
    "vitocm_mim_backward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_size_t, c_void_p]),
    "vitocm_mim_backward_events": (c_int, [c_void_p, c_void_p, c_int]),
    "vitocm_encoder_train_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_size_t,
                                             c_void_p]),
    "vitocm_encoder_backward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_size_t, c_void_p]),
    "vitocm_stream_wait_event": (c_int, [c_void_p, c_void_p]),
    "vitocm_grad_sumsq": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "vitocm_grad_clip": (c_int, [c_void_p, c_int64, c_float, c_void_p, c_void_p]),
    "vitocm_adamw_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float, c_float, c_float, c_float,
                                  c_int, c_float, c_float, c_void_p, c_void_p]),
    "vitocm_wgrad": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "vitocm_attention_fwd_lse": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    "vitocm_attention_bwd": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_int64, c_int, c_int, c_void_p]),
    "vitocm_gemm_dgelu": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_int64, c_void_p,
                                  c_int64, c_void_p]),
    "vitocm_layernorm_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_int, c_int, c_int, c_void_p, c_void_p]),
    "vitocm_mim_loss_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                                    c_void_p]),
    "vitocm_debug_abw_timeline": (c_int, [c_void_p]),
    "vitocm_launch_count": (c_int64, []),
    "vitocm_profile_enable": (c_int, [c_int]),
    "vitocm_profile_classes": (c_int, []),
    "vitocm_profile_class_name": (c_char_p, [c_int]),
    "vitocm_profile_read": (c_int, [c_void_p, c_void_p, c_int]),
}

_lib = None


class VitocmError(RuntimeError):
    pass


def load_library() -> C.CDLL:
    """dlopen libvitocm.so and declare every exported symbol.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VitocmError(f"{LIB_PATH} not found: build it with `python {os.path.join(PKG_DIR, 'build.py')}` "
                          "(nvcc, sm_100a).  There is no CPU / PyTorch fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load_library().vitocm_last_error()
        raise VitocmError(f"libvitocm error {rc}: {msg.decode() if msg else ''}")


def ptr(t) -> int | None:
    """Device (or host) address of a tensor; None passes NULL."""
    if t is None:
        return None
    assert t.is_contiguous(), "vitocm expects dense row-major tensors"
    return t.data_ptr()


def cur_stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def profile_enable(on: bool) -> None:
    load_library().vitocm_profile_enable(int(on))


def profile_read() -> dict:
    """{class name: (total ms, launches)} since the last read."""
    lib = load_library()
    n = lib.vitocm_profile_classes()
    ms = (C.c_double * n)()
    cnt = (C.c_int64 * n)()
    check(lib.vitocm_profile_read(ms, cnt, n))
    return {lib.vitocm_profile_class_name(i).decode(): (float(ms[i]), int(cnt[i])) for i in range(n)}


def launch_count() -> int:
    return int(load_library().vitocm_launch_count())
