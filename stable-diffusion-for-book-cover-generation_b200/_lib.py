"""ctypes binding of libb200sd.so (include/b200sd.h).  There is NO fallback: a missing library or a
failing call raises -- the product path never routes through PyTorch eager or the oracle."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200sd.so")

_lib = None


class B200SDError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [
        ("a0", C.c_void_p), ("a1", C.c_void_p), ("w", C.c_void_p), ("bias", C.c_void_p), ("rowbias", C.c_void_p),
        ("residual", C.c_void_p), ("out", C.c_void_p),
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int), ("C0", C.c_int), ("C1", C.c_int),
        ("lda0", C.c_int), ("lda1", C.c_int), ("ldc", C.c_int), ("ldr", C.c_int), ("ldrb", C.c_int), ("conv_taps", C.c_int),
        ("batch", C.c_int), ("H", C.c_int), ("W", C.c_int), ("rows_per_image", C.c_int), ("epilogue", C.c_int),
        ("out_dtype", C.c_int), ("residual_dtype", C.c_int), ("block_n", C.c_int), ("split_k", C.c_int),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t), ("pair", C.c_int), ("gn_part", C.c_void_p),
    ]


class DgradArgs(C.Structure):
    _fields_ = [
        ("dy", C.c_void_p), ("w", C.c_void_p), ("residual", C.c_void_p), ("out", C.c_void_p),
        ("M", C.c_int), ("Cout", C.c_int), ("Cin", C.c_int), ("conv_taps", C.c_int),
        ("batch", C.c_int), ("H", C.c_int), ("W", C.c_int), ("ldy", C.c_int), ("ldc", C.c_int), ("ldr", C.c_int),
        ("out_dtype", C.c_int), ("residual_dtype", C.c_int), ("block_n", C.c_int), ("pair", C.c_int),
    ]


class WgradArgs(C.Structure):
    _fields_ = [
        ("dy", C.c_void_p), ("x", C.c_void_p), ("dw", C.c_void_p),
        ("rows", C.c_int), ("Cout", C.c_int), ("Cin", C.c_int), ("conv_taps", C.c_int),
        ("batch", C.c_int), ("H", C.c_int), ("W", C.c_int), ("ldy", C.c_int), ("ldx", C.c_int), ("lddw", C.c_int),
        ("block_n", C.c_int), ("split_k", C.c_int),
    ]


_vp, _i, _i64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t

# name -> (restype, argtypes); must list EVERY symbol include/b200sd.h declares (tests check this)
SIGNATURES = {
    "b200sd_last_error": (C.c_char_p, []),
    "b200sd_version": (_i, []),
    "b200sd_launch_count": (_i64, []),
    "b200sd_debug_set": (None, [_i, _i]),
    "b200sd_timer_reserve": (_i, [_i]),
    "b200sd_timer_record": (_i, [_i, _vp]),
    "b200sd_timer_elapsed_ms": (_i, [_i, _i, C.POINTER(C.c_float)]),
    "b200sd_cfg_ddim_step": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _f, _f, _f, _f, _f, _i, _i, _vp]),
    "b200sd_clip_embed": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "b200sd_clip_embed_bwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "b200sd_quick_gelu_fwd": (_i, [_vp, _vp, _i64, _vp]),
    "b200sd_quick_gelu_bwd": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "b200sd_layernorm_f32out": (_i, [_vp, _vp, _vp, _vp, _i, _i, _f, _vp]),
    "b200sd_causal_attention": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "b200sd_causal_attention_bwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "b200sd_im2col_s2_pad": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "b200sd_softmax_rows": (_i, [_vp, _vp, _i, _i, _i, _i, _f, _vp]),
    "b200sd_conv1x1_small": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "b200sd_gaussian_sample": (_i, [_vp, _vp, _vp, _i, _i, _i, _f, _vp]),
    "b200sd_sampler_advance": (_i, [_vp, _i, _vp, _vp, _i, _vp]),
    "b200sd_cfg_plms_step_table": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _f, _vp, _vp, _vp]),
    "b200sd_cfg_ancestral_step": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _f, _f, _f, _f, _f, _f, _f, _i, _i, _i, _vp]),
    "b200sd_cfg_ancestral_step_table": (_i, [_vp, _vp, _vp, _vp, _i64, _f, _vp, _vp, _vp]),
    "b200sd_cfg_plms_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, C.POINTER(C.c_float), _i64, _f, _f,
                                  _f, _i, _i, _vp]),
    "b200sd_add_noise": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i, _i, _vp]),
    "b200sd_inpaint_blend": (_i, [_vp, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _i, _vp]),
    "b200sd_inpaint_blend_table": (_i, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _i, _vp]),
    "b200sd_mse_workspace_floats": (_i, []),
    "b200sd_mse_loss_fwd": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _vp]),
    "b200sd_mse_loss_bwd": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _vp]),
    "b200sd_timestep_embedding": (_i, [_vp, _vp, _i, _i, _vp]),
    "b200sd_small_linear": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200sd_gemm_workspace_bytes": (_sz, []),
    "b200sd_geglu_tile": (_i, [_i]),
    "b200sd_gemm": (_i, [C.POINTER(GemmArgs), _vp]),
    "b200sd_gemm_gn_layout": (_i, [C.POINTER(GemmArgs), _i, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "b200sd_groupnorm_silu_parts": (_i, [_vp, _vp, _i, _i, _vp, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _i,
                                         _i, _vp]),
    "b200sd_gemm_dgrad": (_i, [C.POINTER(DgradArgs), _vp]),
    "b200sd_gemm_wgrad": (_i, [C.POINTER(WgradArgs), _vp]),
    "b200sd_conv_in": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "b200sd_conv_out": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200sd_nhwc_bias_to_nchw": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "b200sd_groupnorm_silu": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _i, _i, _vp]),
    "b200sd_groupnorm_silu_stats": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _i, _i, _vp]),
    "b200sd_groupnorm_workspace_floats": (_i, [_i]),
    "b200sd_layernorm": (_i, [_vp, _vp, _vp, _vp, _i, _i, _f, _i, _vp]),
    "b200sd_attention_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "b200sd_attention": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp, _sz, _vp]),
    "b200sd_attention_lse": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp, _sz, _vp]),
    "b200sd_attention_bwd_workspace_bytes": (_sz, [_i, _i, _i]),
    "b200sd_attention_bwd": (_i, [_vp] * 9 + [_i] * 13 + [_f, _vp, _sz, _vp]),
    "b200sd_grad_prep": (_i, [_vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200sd_groupnorm_bwd_workspace_floats": (_i, [_i]),
    "b200sd_groupnorm_silu_bwd": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _i,
                                       _i, _i, _f, _i, _vp]),
    "b200sd_layernorm_bwd": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp]),
    "b200sd_geglu_fwd": (_i, [_vp, _vp, _i64, _i, _vp]),
    "b200sd_geglu_bwd": (_i, [_vp, _vp, _vp, _i64, _i, _vp]),
    "b200sd_upsample2x_bwd": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200sd_col2im_s2": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200sd_conv_out_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200sd_conv_in_wgrad": (_i, [_vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200sd_cast_act": (_i, [_vp, _vp, _i64, _i, _vp]),
    "b200sd_silu_bwd_mul": (_i, [_vp, _vp, _i64, _vp]),
    "b200sd_split_hi_lo": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "b200sd_groupnorm_silu_split": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _i, _i, _vp]),
    "b200sd_layernorm_split": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _f, _i, _vp]),
    "b200sd_geglu_f32": (_i, [_vp, _vp, _vp, _i64, _i, _vp]),
    "b200sd_attention_f32": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "b200sd_small_linear_f32": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200sd_cast_flat": (_i, [_vp, _vp, _i64, _vp]),
    "b200sd_adamw_step": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _f, _f, _f, _f, _f, _i, _f, _i, _vp]),
    "b200sd_adamw8bit_step": (_i, [_vp] * 12 + [_i64, _f, _f, _f, _f, _f, _i, _f, _i, _vp]),
    "b200sd_upsample2x": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200sd_im2col_s2": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
}


def lib() -> C.CDLL:
    """Load (once) and return the CUDA library; raise loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200SDError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(b200sd has no CPU / eager fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().b200sd_last_error().decode("utf-8", "replace")
        raise B200SDError(f"{what or 'b200sd call'} failed (code {rc}): {msg}")
