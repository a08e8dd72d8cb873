"""ctypes binding of the C-ABI library ``libw2s.so`` (include/w2s.h).

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  There is no
Python/CPU implementation behind it: if the shared object is missing, or no B200 is present
when a handle is created, the error is raised to the caller.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libw2s.so")

MAX_CONV_LAYERS = 8

OUT_MAX, OUT_LOGIT, OUT_LOGPROB, OUT_MEAN, OUT_LOGITS, OUT_CTC, OUT_ERRORS = 0, 1, 2, 3, 4, 5, 6
ERR_UNITS = {"labels": 0, "words": 1}     # W2S_ERR_LABELS / W2S_ERR_WORDS (OUT_ERRORS, set by w2s_set_references only)
MODE_IDS = {"max": OUT_MAX, "logit": OUT_LOGIT, "logprob": OUT_LOGPROB, "mean": OUT_MEAN, "logits": OUT_LOGITS}
FLAG_VALIDATE_GEMM, FLAG_VALIDATE_ATTN, FLAG_FP32_PRELN, FLAG_NO_GRAPH, FLAG_DENSE_FRONTEND = 1, 2, 4, 16, 32
MAX_BACKGROUND = 256      # W2S_MAX_BACKGROUND: rows of a background set
MAX_BANDS = 16            # W2S_MAX_BANDS: frequency bands of time-frequency cells
MAX_TRANSCRIPT = 512      # W2S_MAX_TRANSCRIPT: labels of one transcript (OUT_CTC, set by w2s_set_transcripts only)


class W2SConfig(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("num_conv_layers", C.c_int32),
        ("conv_dim", C.c_int32 * MAX_CONV_LAYERS),
        ("conv_kernel", C.c_int32 * MAX_CONV_LAYERS),
        ("conv_stride", C.c_int32 * MAX_CONV_LAYERS),
        ("conv_bias", C.c_int32),
        ("feat_extract_norm", C.c_int32),
        ("hidden_size", C.c_int32),
        ("num_hidden_layers", C.c_int32),
        ("num_attention_heads", C.c_int32),
        ("intermediate_size", C.c_int32),
        ("num_conv_pos_embeddings", C.c_int32),
        ("num_conv_pos_embedding_groups", C.c_int32),
        ("vocab_size", C.c_int32),
        ("layer_norm_eps", C.c_float),
        ("do_stable_layer_norm", C.c_int32),
        ("position_embeddings_type", C.c_int32),
        ("conv_depthwise_kernel_size", C.c_int32),
        ("hidden_act", C.c_int32),
        ("rotary_embedding_base", C.c_int32),
        ("max_batch", C.c_int32),
        ("flags", C.c_int32),
        ("num_buckets", C.c_int32),
        ("max_bucket_distance", C.c_int32),
    ]


# every symbol include/w2s.h declares: (restype, argtypes)
SIGNATURES = {
    "w2s_create": (C.c_int, [C.POINTER(W2SConfig), C.POINTER(C.c_char_p), C.POINTER(C.c_void_p),
                             C.POINTER(C.c_int64), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "w2s_destroy": (None, [C.c_void_p]),
    "w2s_last_error": (C.c_char_p, [C.c_void_p]),
    "w2s_num_frames": (C.c_int64, [C.c_void_p, C.c_int64]),
    "w2s_set_clip": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int32), C.c_int, C.c_float,
                               C.c_void_p]),
    "w2s_set_background": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.POINTER(C.c_double),
                                     C.c_void_p]),
    "w2s_set_bands": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p]),
    "w2s_set_targets": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int, C.c_int,
                                  C.c_void_p]),
    "w2s_set_transcripts": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int, C.c_int,
                                      C.c_void_p]),
    "w2s_set_references": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_void_p]),
    "w2s_out_width": (C.c_int64, [C.c_void_p, C.c_int64]),
    "w2s_eval": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "w2s_eval_waveforms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                     C.c_void_p]),
    "w2s_grad_waveforms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.POINTER(C.c_int32),
                                     C.c_void_p, C.c_void_p, C.c_void_p]),
    "w2s_vjp_waveforms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]),
    "w2s_grad_transcripts": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.POINTER(C.c_int32),
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "w2s_grad_debug": (C.c_int, [C.c_void_p, C.c_int]),
    "w2s_grad_rules": (C.c_int, [C.c_void_p, C.c_int]),
    "w2s_grad_peek": (C.c_int64, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "w2s_mask": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "w2s_wls": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p,
                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "w2s_sample_rows": (C.c_int64, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "w2s_relative_buckets": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "w2s_frontend_blocks": (C.c_int64, [C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p,
                                        C.c_int64]),
    "w2s_debug_gemm": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float,
                                 C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "w2s_debug_attention": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p,
                                      C.c_void_p, C.c_void_p]),
    "w2s_debug_attention_bias": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float,
                                           C.c_void_p, C.c_void_p, C.c_void_p]),
    "w2s_debug_attention_bwd": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                          C.c_float, C.c_void_p, C.c_void_p]),
    "w2s_debug_ctc": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                C.c_int, C.c_int, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p, C.c_void_p]),
    "w2s_debug_errors": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                   C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "w2s_error_tables": (C.c_int64, [C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_void_p, C.c_int64]),
    "w2s_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "w2s_profile_read": (C.c_int64, [C.c_void_p, C.c_char_p, C.c_int64, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                     C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int64]),
    "w2s_kernel_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "w2s_launch_count": (C.c_int64, [C.c_void_p]),
    "w2s_flops_per_forward": (C.c_double, [C.c_void_p, C.c_int64]),
}

_lib = None


def load():
    """Load libw2s.so and bind every declared entry point; raises if the build is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()'). "
            "There is no CPU fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
