"""ctypes binding of libhh_b200.so (declarations: include/hh_b200.h).

There is no CPU or PyTorch fallback behind these calls: if the shared library is missing, or a call is made with
tensors that are not on a CUDA device, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# HH_B200_LIB: developer override to A/B two builds of the same library on one GPU box (never a different backend)
LIB_PATH = os.environ.get("HH_B200_LIB") or os.path.join(_HERE, "libhh_b200.so")


class EncoderCfg(C.Structure):
    _fields_ = [(k, C.c_int) for k in ("img_size", "patch_size", "num_frames", "embed_dim", "depth", "num_heads",
                                       "mlp_hidden")]


class DecoderCfg(C.Structure):
    _fields_ = [(k, C.c_int) for k in ("d_model", "nhead", "num_layers", "dim_feedforward", "num_queries",
                                       "num_classes1", "feature_dim", "num_frames", "patches_per_frame", "pred_traj")]


class TextCfg(C.Structure):
    _fields_ = [(k, C.c_int) for k in ("vocab_size", "context_length", "width", "heads", "layers", "embed_dim")]


_p, _i, _f, _i64, _sz = C.c_void_p, C.c_int, C.c_float, C.c_int64, C.c_size_t

# name -> (restype, argtypes); must list every symbol include/hh_b200.h declares (tests/test_capi_symbols.py checks)
SIGNATURES = {
    "hh_last_error": (C.c_char_p, []),
    "hh_version": (_i, []),
    "hh_encoder_create": (_i, [C.POINTER(_p), C.POINTER(EncoderCfg)]),
    "hh_encoder_destroy": (None, [_p]),
    "hh_encoder_set_weight": (_i, [_p, C.c_char_p, _p, _i64, _p]),
    "hh_encoder_forward": (_i, [_p, _p, _i, _p, _p]),
    "hh_encoder_forward_n": (_i, [_p, _p, _i, _i, _p, _p]),
    "hh_encoder_forward_u8": (_i, [_p, _p, _i, C.POINTER(_f), C.POINTER(_f), _p, _p]),
    "hh_encoder_forward_bf16": (_i, [_p, _p, _i, _p, _p, _p]),
    "hh_encoder_forward_u8_bf16": (_i, [_p, _p, _i, C.POINTER(_f), C.POINTER(_f), _p, _p, _p]),
    "hh_encoder_flops_per_clip": (C.c_double, [_p]),
    "hh_encoder_last_launches": (_i, [_p]),
    "hh_decoder_create": (_i, [C.POINTER(_p), C.POINTER(DecoderCfg)]),
    "hh_decoder_destroy": (None, [_p]),
    "hh_decoder_set_weight": (_i, [_p, C.c_char_p, _p, _i64, _p]),
    "hh_decoder_forward": (_i, [_p, _p, _i64, _i64, _i, _i, _p, _p, _p, _p]),
    "hh_decoder_forward_train": (_i, [_p, _p, _i64, _i64, _i, _i, _p, _p, _p, _p]),
    "hh_decoder_forward_bf16": (_i, [_p, _p, _i64, _i64, _i, _i, _p, _p, _p, _p]),
    "hh_decoder_forward_train_bf16": (_i, [_p, _p, _i64, _i64, _i, _i, _p, _p, _p, _p]),
    "hh_decoder_set_dropout": (_i, [_p, _f, C.c_uint64, C.c_uint32]),
    "hh_decoder_backward": (_i, [_p, _p, _p, _p, _p, _p]),
    "hh_decoder_generation": (C.c_uint64, [_p]),
    "hh_decoder_backward_checked": (_i, [_p, C.c_uint64, _p, _p, _p, _p, _p]),
    "hh_decoder_get_grad": (_i, [_p, C.c_char_p, _p, _i64, _p]),
    "hh_decoder_get_grads": (_i, [_p, _p, _p, _i, _p, _i64, _p]),
    "hh_decoder_get_saved": (_i, [_p, C.c_char_p, _i, _p, _i64, _p]),
    "hh_decoder_set_weights": (_i, [_p, _p, _p, _p, _i, _p]),
    "hh_decoder_flops_per_clip": (C.c_double, [_p, _i]),
    "hh_decoder_last_launches": (_i, [_p]),
    "hh_text_create": (_i, [C.POINTER(_p), C.POINTER(TextCfg)]),
    "hh_text_destroy": (None, [_p]),
    "hh_text_set_weight": (_i, [_p, C.c_char_p, _p, _i64, _p]),
    "hh_text_forward": (_i, [_p, _p, _i, _p, _p, _p]),
    "hh_text_flops_per_sequence": (C.c_double, [_p]),
    "hh_text_last_launches": (_i, [_p]),
    "hh_box_loss_forward": (_i, [_p, _p, _p, _i, _f, _p, _p]),
    "hh_box_loss_backward": (_i, [_p, _p, _p, _i, _f, _p, _p, _i64, _p]),
    "hh_assign": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _p, _p, _p, _i, _p]),
    "hh_match_cost_class": (_i, [_p, _i, _i, _p, _i, _f, _p, _p]),
    "hh_sim_matrix_backward_workspace_bytes": (_sz, [_i, _i]),
    "hh_sim_matrix_backward": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _f, _p, _p]),
    "hh_egonce_forward": (_i, [_p, _i, _i, _p, _p, _i, _p, _f, _f, _p, _p, _p, _p]),
    "hh_egonce_backward": (_i, [_p, _i, _i, _f, _p, _p, _p, _p, _p, _p]),
    "hh_word_loss_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "hh_word_loss_forward": (_i, [_p, _i, _i, _p, _i, _i, _p, _i, _f, _f, _p, _p, _p, _p, _p, _p, _p]),
    "hh_word_loss_backward": (_i, [_p, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "hh_retrieval_rows": (_i, [_p, _p, _p, _p, _i, _i, _i, _p, _p]),
    "hh_linear_f32_backward": (_i, [_p, _i, _p, _i, _i, _p, _p, _i, _p, _i, _i, _p, _i, _p, _p, _i, _i, _i, _f, _f, _p]),
    "hh_layernorm_backward": (_i, [_p, _i, _p, _f, _p, _i, _p, _p, _p, _i, _i, _p]),
    "hh_self_attention_backward": (_i, [_p, _p, _p, _i, _p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "hh_cross_attention_backward": (_i, [_p, _p, _p, _i, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "hh_attention_causal": (_i, [_p, _p, _i, _i, _i, _p]),
    "hh_profile_num_classes": (_i, []),
    "hh_profile_class_name": (C.c_char_p, [_i]),
    "hh_encoder_set_profile": (_i, [_p, _i]),
    "hh_encoder_profile": (_i, [_p, C.POINTER(C.c_double), C.POINTER(_i)]),
    "hh_decoder_set_profile": (_i, [_p, _i]),
    "hh_decoder_profile": (_i, [_p, C.POINTER(C.c_double), C.POINTER(_i)]),
    "hh_sim_matrix": (_i, [_p, _p, _p, _i, _i, _i, _f, _p]),
    "hh_row_reduce": (_i, [_p, _i, _i, _f, _i, _p, _p]),
    "hh_l2_normalize": (_i, [_p, _p, _i, _i, _f, _p]),
    "hh_linear_f32": (_i, [_p, _i, _p, _i, _p, _p, _p, _i, _p, _i, _i, _i, _i, _i, _i, _p]),
    "hh_box_cxcywh_to_xyxy": (_i, [_p, _p, _i64, _p]),
    "hh_box_xyxy_to_cxcywh": (_i, [_p, _p, _i64, _p]),
    "hh_box_pairwise": (_i, [_p, _p, _i, _i, _p, _p, _p, _p]),
    "hh_box_match_cost": (_i, [_p, _p, _i, _i, _f, _f, _p, _p]),
    "hh_gemm_bf16": (_i, [_p, _i, _p, _i, _p, _i, _p, _p, _i, _i, _i, _i, _i, _p]),
    "hh_gemm_stats_parts": (_i, [_i, _i]),
    "hh_fold_layernorm_weight": (_i, [_p, _p, _p, _p, _i, _i, _i, _f, _p, _p, _p, _p]),
    "hh_gemm_bf16_res_stats": (_i, [_p, _i, _p, _i, _p, _i, _p, _p, _i, _i, _p, _i, _i, _i, _p]),
    "hh_gemm_bf16_ln": (_i, [_p, _i, _p, _i, _p, _i, _p, _p, _p, _i, _i, _f, _i, _i, _i, _i, _p]),
    "hh_layernorm": (_i, [_p, _i, _p, _p, _f, _p, _p, _i, _i, _p]),
    "hh_f32_to_bf16": (_i, [_p, _p, _i64, _p]),
    "hh_attention": (_i, [_p, _p, _i, _i, _i, _i, _i, _p]),
    "hh_cross_attention": (_i, [_p, _p, _p, _i, _p, _i, _i, _i, _i, _p]),
    "hh_cross_attention_simt": (_i, [_p, _p, _p, _i, _p, _i, _i, _i, _i, _p]),
    "hh_comm_unique_id": (_i, [_p]),
    "hh_comm_create": (_i, [C.POINTER(_p), _i, _i, _p]),
    "hh_comm_destroy": (_i, [_p]),
    "hh_allgather": (_i, [_p, _p, _p, _sz, _p]),
}

_lib = None


def load():
    """Load libhh_b200.so (built by `__graft_entry__.build()` / `make -C .../csrc`). Fails loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            "libhh_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` at the repo "
            "root. There is no CPU/PyTorch fallback for this path." % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    msg = load().hh_last_error()
    return msg.decode() if msg else ""


def check(rc: int, what: str):
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (what, rc, last_error()))


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t: torch.Tensor | None) -> int | None:
    """Device pointer of a contiguous CUDA tensor (None passes NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("helping_hand_for_egocentric_videos_b200: tensor is on %s; this path only runs on CUDA "
                           "(no CPU fallback)" % t.device)
    if not t.is_contiguous():
        raise RuntimeError("helping_hand_for_egocentric_videos_b200: tensor must be contiguous")
    return t.data_ptr()


def require_f32(t: torch.Tensor, name: str):
    if t.dtype != torch.float32:
        raise RuntimeError("%s must be float32, got %s" % (name, t.dtype))
