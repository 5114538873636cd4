"""ctypes binding of libgitb200.so (the C ABI declared in include/gitb200.h).

There is no fallback: if the shared library is missing or cannot be loaded, importing the engine
raises.  The library is built in-tree by ``build.py`` (``__graft_entry__.build()``)."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_int64, c_longlong, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgitb200.so")


class GitB200Error(RuntimeError):
    pass


class Config(Structure):
    _fields_ = [
        ("vit_width", c_int), ("vit_layers", c_int), ("vit_heads", c_int), ("patch", c_int), ("resolution", c_int),
        ("hidden", c_int), ("dec_layers", c_int), ("dec_heads", c_int), ("ffn", c_int),
        ("vocab", c_int), ("max_positions", c_int),
        ("num_image_with_embedding", c_int),
        ("vit_ln_eps", c_float), ("proj_ln_eps", c_float), ("embed_ln_eps", c_float), ("bert_ln_eps", c_float),
        ("sos", c_int), ("eos", c_int),
    ]


class StudentConfig(Structure):
    _fields_ = [
        ("d_model", c_int), ("n_head", c_int), ("d_ffn", c_int), ("n_layers", c_int),
        ("vocab", c_int), ("max_len", c_int), ("cls", c_int), ("sep", c_int), ("pad", c_int), ("ln_eps", c_float),
    ]


class SearchParams(Structure):
    _fields_ = [
        ("beam_size", c_int), ("max_steps", c_int), ("per_node_beam_size", c_int), ("num_keep_best", c_int),
        ("length_penalty", c_float), ("reorder_cache", c_int),
    ]


# name -> (restype, argtypes); must list every symbol include/gitb200.h declares (tests check this)
SIGNATURES = {
    "gitb200_create": (c_int, [POINTER(Config), c_int, POINTER(c_void_p)]),
    "gitb200_destroy": (None, [c_void_p]),
    "gitb200_last_error": (c_char_p, [c_void_p]),
    "gitb200_version": (c_char_p, []),
    "gitb200_load_weight": (c_int, [c_void_p, c_char_p, c_void_p, c_int, POINTER(c_int64)]),
    "gitb200_finalize_weights": (c_int, [c_void_p]),
    "gitb200_reserve": (c_int, [c_void_p, c_int, c_int, c_int, c_int]),
    "gitb200_tokens_per_frame": (c_int, [c_void_p]),
    "gitb200_logits_ld": (c_int, [c_void_p]),
    "gitb200_encode": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "gitb200_student_create": (c_int, [POINTER(StudentConfig), c_int, POINTER(c_void_p)]),
    "gitb200_student_destroy": (None, [c_void_p]),
    "gitb200_student_last_error": (c_char_p, [c_void_p]),
    "gitb200_student_load_weight": (c_int, [c_void_p, c_char_p, c_void_p, c_int, POINTER(c_int64)]),
    "gitb200_student_finalize": (c_int, [c_void_p]),
    "gitb200_student_set_training": (c_int, [c_void_p, c_int]),
    "gitb200_student_train_begin": (c_longlong, [c_void_p, c_float, c_float, c_float, c_float]),
    "gitb200_student_train_head_floats": (c_longlong, [c_void_p]),
    "gitb200_student_train_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "gitb200_student_train_backward": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "gitb200_student_train_apply": (c_int, [c_void_p, c_void_p, c_float, c_void_p]),
    "gitb200_student_train_export": (c_int, [c_void_p, c_char_p, c_int, c_void_p, c_void_p, c_void_p]),
    "gitb200_student_logits_ld": (c_int, [c_void_p]),
    "gitb200_student_forward_decoder": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "gitb200_student_greedy_decode": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "gitb200_encode_images": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "gitb200_set_vit_taps": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "gitb200_set_visual_features": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "gitb200_decode": (c_int, [c_void_p, POINTER(SearchParams), c_void_p, c_void_p, c_void_p, c_void_p]),
    "gitb200_caption": (c_int, [c_void_p, c_void_p, c_int, c_int, POINTER(SearchParams), c_void_p, c_void_p, c_void_p,
                                c_void_p]),
    "gitb200_set_fold_layernorm": (c_int, [c_void_p, c_int]),
    "gitb200_set_pipeline": (c_int, [c_void_p, c_int]),
    "gitb200_caption_from_host": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, POINTER(SearchParams), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gitb200_set_early_exit": (c_int, [c_void_p, c_int]),
    "gitb200_set_persistent_decode": (c_int, [c_void_p, c_int]),
    "gitb200_debug_persistent_decode_trace": (c_int, [c_void_p, c_void_p, c_int]),
    "gitb200_last_decode_steps": (c_int, [c_void_p]),
    "gitb200_set_graph_max_clips": (c_int, [c_void_p, c_int]),
    "gitb200_set_graph_segments": (c_int, [c_void_p, c_int]),
    "gitb200_set_fuse_layernorm": (c_int, [c_void_p, c_int]),
    "gitb200_op_gemm_ln": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p]),
    "gitb200_set_sweep_rows": (c_int, [c_void_p, c_int]),
    "gitb200_caption_host": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, POINTER(SearchParams), c_void_p, c_void_p]),
    "gitb200_caption_host_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, POINTER(SearchParams), c_void_p,
                                        c_void_p]),
    "gitb200_forward_logits": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                       c_void_p]),
    "gitb200_decode_begin": (c_int, [c_void_p, c_int, c_void_p]),
    "gitb200_decode_step": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "gitb200_decode_reorder": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "gitb200_stream_reset": (c_int, [c_void_p]),
    "gitb200_stream_push": (c_int, [c_void_p, c_void_p, c_void_p]),
    "gitb200_stream_push_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "gitb200_stream_frames": (c_int, [c_void_p]),
    "gitb200_stream_caption": (c_int, [c_void_p, POINTER(SearchParams), c_void_p, c_void_p, c_void_p]),
    "gitb200_streams_configure": (c_int, [c_void_p, c_int]),
    "gitb200_streams_push": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "gitb200_streams_push_u8": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_void_p]),
    "gitb200_streams_caption": (c_int, [c_void_p, c_void_p, c_int, POINTER(SearchParams), c_void_p, c_void_p, c_void_p]),
    "gitb200_streams_reset": (c_int, [c_void_p, c_void_p, c_int]),
    "gitb200_streams_frames": (c_int, [c_void_p, c_int]),
    "gitb200_streams_window": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "gitb200_preprocess": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "gitb200_op_gemm": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                c_int, c_void_p]),
    "gitb200_op_layernorm": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_float, c_void_p, c_void_p]),
    "gitb200_op_attention_groups": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p]),
    "gitb200_op_text_attention": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "gitb200_op_attention_groups_mma": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p]),
    "gitb200_op_search": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, POINTER(SearchParams), c_void_p, c_void_p,
                                  c_void_p]),
    "gitb200_launch_count": (c_longlong, [c_int]),
    "gitb200_graph_launches": (c_longlong, [c_void_p]),
    "gitb200_profile_gemm": (None, [c_int]),
    "gitb200_profile_gemm_read": (None, [POINTER(ctypes.c_double), POINTER(ctypes.c_double), POINTER(c_longlong)]),
    "gitb200_profile_decode_attention_read": (None, [POINTER(ctypes.c_double), POINTER(ctypes.c_double), POINTER(c_longlong)]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load libgitb200.so and declare every entry point.  Raises GitB200Error if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GitB200Error(
            f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` (nvcc, sm_100a). "
            "gitb200 has no CPU / PyTorch fallback path.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, ctx=None, what: str = "") -> None:
    if rc != 0:
        msg = load().gitb200_last_error(ctx)
        raise GitB200Error(f"{what} failed with status {rc}: {msg.decode() if msg else '?'}")
