"""ctypes binding of ``liblavie_b200.so`` (the C ABI declared in include/lavie_b200.h).

There is deliberately NO fallback: if the shared object is missing or an entry point returns an
error the caller gets an exception, never a PyTorch re-implementation.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_longlong, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LAVIE_LIB_PATH") or os.path.join(_HERE, "liblavie_b200.so")   # override: A/B of two builds


class LavieError(RuntimeError):
    pass


class Epilogue(Structure):
    """mirror of ``lavie_epilogue``"""
    _fields_ = [
        ("bias", c_void_p),
        ("row_bias", c_void_p),
        ("ld_row_bias", c_int),
        ("rows_per_batch", c_int),
        ("residual", c_void_p),
        ("ld_residual", c_int),
        ("geglu", c_int),
        ("col_stats", c_void_p),
    ]


# name -> (restype, argtypes); must list every symbol declared in include/lavie_b200.h
_P = c_void_p
SIGNATURES = {
    "lavie_last_error": (c_char_p, []),
    "lavie_abi_version": (c_int, []),
    "lavie_debug_set": (c_int, [c_int, c_int]),
    "lavie_debug_buffer": (c_int, [c_void_p]),
    "lavie_gemm_plan": (c_int, [c_int, c_int, c_int, c_int, c_int, c_size_t, POINTER(c_int), POINTER(c_int),
                                POINTER(c_int), POINTER(c_int)]),
    "lavie_gemm_bf16": (c_int, [_P, c_int, c_int, _P, c_int, c_int, _P, _P, c_int, c_int, c_int, POINTER(Epilogue),
                                c_int, _P, c_size_t, _P]),
    "lavie_conv3x3_supported": (c_int, [c_int, c_int, c_int]),
    "lavie_conv3x3_bf16": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, c_int, POINTER(Epilogue), c_int, _P,
                                   c_size_t, _P]),
    "lavie_conv3x3_pad_bf16": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, c_int,
                                       POINTER(Epilogue), c_int, _P, c_size_t, _P]),
    "lavie_conv3x3_out_size": (c_int, [c_int, c_int, c_int, c_int]),
    "lavie_im2col3x3_bf16": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "lavie_groupnorm_chunks": (c_int, [c_int, c_int]),
    "lavie_groupnorm_stats": (c_int, [_P, c_int, c_int, _P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "lavie_groupnorm_finalize": (c_int, [_P, c_int, c_int, c_int, c_int, c_longlong, _P, _P, c_float, _P, _P]),
    "lavie_groupnorm_scale_shift": (c_int, [_P, c_int, c_int, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_float,
                                            _P, _P, _P, _P]),
    "lavie_groupnorm_finalize_colsums": (c_int, [_P, c_int, _P, c_int, c_int, c_int, c_int, _P, _P, c_float, _P, _P]),
    "lavie_groupnorm_reduce_colsums": (c_int, [_P, c_int, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "lavie_groupnorm_apply": (c_int, [_P, c_int, c_int, _P, c_int, c_int, c_int, c_int, _P, c_int, _P, c_int, _P]),
    "lavie_layernorm_bf16": (c_int, [_P, c_int, _P, _P, c_float, _P, c_int, c_int, c_int, _P]),
    "lavie_layernorm_scatter_bf16": (c_int, [_P, c_int, _P, _P, c_float, _P, c_int, c_int, c_int, c_int, c_int, _P]),
    "lavie_add_gathered_bf16": (c_int, [_P, c_int, _P, c_int, _P, c_int, c_int, c_int, c_int, c_int, _P]),
    "lavie_groupnorm_reduce": (c_int, [_P, c_int, c_int, c_int, _P, _P]),
    "lavie_p2p_fault_buffer": (c_int, [_P, c_int]),
    "lavie_rank_barrier": (c_int, [_P, _P, c_int, c_int, _P]),
    "lavie_gn_exchange_finalize": (c_int, [_P, c_int, c_int, c_int, c_int, c_longlong, _P, _P, c_float, _P, _P, _P, _P,
                                           c_int, c_int, _P]),
    "lavie_gn_exchange_finalize_sums": (c_int, [_P, c_int, c_int, c_int, c_longlong, _P, _P, c_float, _P, _P, _P, _P, c_int,
                                                c_int, _P]),
    "lavie_layernorm_scatter_p2p": (c_int, [_P, c_int, _P, _P, c_float, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                            _P, _P, _P, _P]),
    "lavie_add_gathered_p2p": (c_int, [_P, c_int, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P,
                                       _P, _P]),
    "lavie_halo_push_p2p": (c_int, [_P, _P, c_longlong, _P, c_int, c_int, _P, _P, _P, _P]),
    "lavie_gn_exchange_finalize_colsums": (c_int, [_P, c_int, _P, c_int, c_int, c_int, c_int, c_longlong, _P, _P, c_float,
                                                   _P, _P, _P, _P, c_int, c_int, _P]),
    "lavie_groupnorm_finalize_sums": (c_int, [_P, c_int, c_int, c_int, c_longlong, _P, _P, c_float, _P, _P]),
    "lavie_attention_bf16": (c_int, [_P, c_int, _P, c_int, _P, c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int,
                                     c_int, c_int, c_float, _P]),
    "lavie_attention_strided_bf16": (c_int, [_P, c_longlong, c_longlong, _P, _P, c_longlong, c_longlong, _P, c_longlong,
                                             c_longlong, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                             c_float, _P]),
    "lavie_temporal_attention_bf16": (c_int, [_P, c_int, c_int, c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int,
                                              c_int, c_float, _P, c_int, _P, _P]),
    "lavie_linear_smallm": (c_int, [_P, c_int, c_int, _P, _P, _P, c_int, c_int, c_int, _P]),
    "lavie_timestep_embedding": (c_int, [_P, c_int, c_int, _P, _P]),
    "lavie_conv_in": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, _P, c_int, _P]),
    "lavie_conv_in_scaled": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, _P, c_int, _P]),
    "lavie_conv_out": (c_int, [_P, c_int, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, _P, _P]),
    "lavie_embedding_add": (c_int, [_P, _P, _P, c_int, c_int, c_int, _P]),
    "lavie_frame_conv_bf16": (c_int, [_P, c_int, c_longlong, c_int, c_int, c_int, _P, _P, c_int, c_int, c_int,
                                      POINTER(Epilogue), c_int, _P, c_size_t, _P]),
    "lavie_clip_embed": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "lavie_causal_attention_small": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_float, _P, c_int, _P]),
    "lavie_activation_bf16": (c_int, [_P, c_longlong, c_int, _P]),
    "lavie_softmax_rows_bf16": (c_int, [_P, c_int, c_longlong, c_int, c_float, _P]),
    "lavie_attention_wide_bf16": (c_int, [_P, c_int, _P, c_int, _P, c_int, _P, c_int, c_int, c_int, _P]),
    "lavie_image_to_uint8": (c_int, [_P, c_int, c_longlong, _P, _P]),
    "lavie_im2col_frames_bf16": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P]),
    "lavie_posterior_sample_f32": (c_int, [_P, _P, c_int, c_int, c_longlong, c_float, _P, _P]),
    "lavie_pointwise_conv_nchw_f32": (c_int, [_P, _P, _P, c_float, c_int, c_int, c_int, c_longlong, _P, _P]),
    "lavie_groupnorm_finalize_colsums_seg": (c_int, [_P, c_int, c_int, _P, c_int, c_int, c_int, c_int, c_int, _P, _P,
                                                     c_float, _P, _P]),
    "lavie_upsample_conv3x3_supported": (c_int, [c_int, c_int, c_int]),
    "lavie_upsample_conv3x3_bf16": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, c_int, POINTER(Epilogue), c_int, _P]),
    "lavie_im2col_input_bf16": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "lavie_unpack_nchw_f32": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "lavie_upsample_nearest2x": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P]),
    "lavie_cfg_ddim_step": (c_int, [_P, _P, c_float, c_float, c_float, _P, _P, c_longlong, _P]),
    "lavie_cfg_linear_step": (c_int, [_P, _P, c_float, c_float, c_float, c_float, _P, _P, _P, c_longlong, _P]),
    "lavie_cfg_combine": (c_int, [_P, _P, c_float, _P, _P, c_longlong, _P]),
    # fp32-accumulate check mode (split-bf16 triples)
    "lavie_check_split3": (c_int, [_P, c_longlong, c_int, _P, _P]),
    "lavie_check_gemm": (c_int, [_P, c_int, c_int, _P, c_int, c_int, _P, _P, c_int, c_int, c_int, POINTER(Epilogue), _P,
                                 c_size_t, _P]),
    "lavie_check_conv3x3": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, c_int, POINTER(Epilogue), _P,
                                    c_size_t, _P]),
    "lavie_check_groupnorm_stats": (c_int, [_P, c_int, c_int, _P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "lavie_check_groupnorm_apply": (c_int, [_P, c_int, c_int, _P, c_int, c_int, c_int, c_int, _P, c_int, _P, c_int, _P]),
    "lavie_check_layernorm": (c_int, [_P, c_int, _P, _P, c_float, _P, c_int, c_int, c_int, _P]),
    "lavie_check_attention": (c_int, [_P, c_longlong, c_longlong, c_int, _P, _P, c_longlong, c_longlong, c_int, _P,
                                      c_longlong, c_longlong, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                      c_int, c_float, _P, c_int, _P, _P]),
    "lavie_check_linear_smallm": (c_int, [_P, c_int, c_int, _P, _P, _P, c_int, c_int, c_int, _P]),
    "lavie_check_conv_in": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, _P, c_int, _P]),
    "lavie_check_conv_out": (c_int, [_P, c_int, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, _P, _P]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load the shared object (once) and bind every declared symbol; raise if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LavieError(
            f"{LIB_PATH} not found: build it with `make` (or __graft_entry__.build()). "
            "lavie_b200 has no CPU / PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if os.environ.get("LAVIE_INKERNEL_SPLITK", "0") == "1":      # A/B switch: in-kernel split-K reduction (slower, off)
        lib.lavie_debug_set(7, 1)
    if os.environ.get("LAVIE_XATTN", "0") == "1":                # A/B switch: text cross-attention on the mma.sync kernel
        lib.lavie_debug_set(8, 1)
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().lavie_last_error()
        raise LavieError(f"{what} failed ({rc}): {msg.decode() if msg else '?'}")
