"""ctypes binding of `csrc/libd3pm_b200.so` (the C ABI declared in `include/d3pm_b200.h`).

There is no fallback: if the library is missing or a call fails, `D3PMError` is raised.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int8, c_int32, c_int64, c_uint32, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_NAME = "libd3pm_b200.so"

# every symbol include/d3pm_b200.h declares (tests check the built library exports exactly these)
EXPORTED_SYMBOLS = (
    "d3pm_version", "d3pm_last_error", "d3pm_build_coef_table", "d3pm_fused_step", "d3pm_philox_uniform",
    "d3pm_q_posterior", "d3pm_gumbel_argmax", "d3pm_tokens_to_log_onehot", "d3pm_argmax_classes",
    "d3pm_to_token_major", "d3pm_q_pred", "d3pm_q_sample_tokens", "d3pm_train_rows", "d3pm_purity_select",
    "d3pm_head_image_floats", "d3pm_head_prepare", "d3pm_head_step", "d3pm_scale_rows",
    "d3pm_decode_lut", "d3pm_tokens_to_features",
    "d3pm_dec_image_floats", "d3pm_dec_weight_image", "d3pm_dec_conv", "d3pm_dec_embed_rows", "d3pm_dec_axial_attention",
    "d3pm_dec_col2im", "d3pm_self_attention",
    "d3pm_host_step_create", "d3pm_host_step_destroy", "d3pm_host_step_h2d_bytes", "d3pm_host_step_d2h_bytes",
    "d3pm_host_step_run", "d3pm_host_head_step_run", "d3pm_host_step_set_logits_dtype",
)

COEF_STRIDE = 32
SAMPLE_NONE, SAMPLE_GUMBEL, SAMPLE_PHILOX, SAMPLE_PHILOX_EXACT = 0, 1, 2, 3
STATUS_BAD_T, STATUS_BAD_TOKEN, STATUS_FALLBACK = 1, 2, 4
KERNEL_AUTO, KERNEL_ROWS, KERNEL_STREAM = 0, 1, 2
FROM_POSTERIOR, FROM_RECON = 0, 1
LOGITS_F32, LOGITS_F16, LOGITS_BF16 = 0, 1, 2
HEAD_STEP, HEAD_LOGITS, HEAD_REFERENCE = 0, 1, 2


class D3PMError(RuntimeError):
    """Raised when libd3pm_b200.so is missing or one of its entry points returns an error."""


class StepDesc(ctypes.Structure):
    """Mirror of `d3pm_step_desc`."""
    _fields_ = [
        ("logits_c", c_void_p), ("logits_u", c_void_p), ("x_t", c_void_p), ("t", c_void_p),
        ("coef_table", c_void_p), ("gumbel", c_void_p),
        ("x_prev", c_void_p), ("post", c_void_p), ("recon", c_void_p), ("gap", c_void_p), ("status", c_void_p),
        ("B", c_int32), ("N", c_int32), ("K", c_int32), ("T", c_int32),
        ("pitch_logits", c_int64), ("pitch_gumbel", c_int64), ("pitch_out", c_int64),
        ("guidance_scale", c_float), ("sample_mode", c_int32), ("gumbel_is_uniform", c_int32),
        ("seed", c_uint64), ("offset", c_uint64), ("row_offset", c_int64),
        ("thin_factor", c_float), ("kernel", c_int32), ("stream", c_void_p),
        ("sample_from", c_int32), ("logits_dtype", c_int32), ("score", c_void_p), ("sharpen", c_void_p),
        ("winner_post", c_void_p),
    ]


class TrainDesc(ctypes.Structure):
    """Mirror of `d3pm_train_desc`."""
    _fields_ = [
        ("logits", c_void_p), ("x0", c_void_p), ("x_t", c_void_p), ("t", c_void_p), ("coef_table", c_void_p),
        ("w_main", c_void_p), ("w_aux", c_void_p), ("tok_main", c_void_p), ("tok_aux", c_void_p),
        ("x0_recon", c_void_p), ("xtm1_recon", c_void_p), ("grad", c_void_p), ("status", c_void_p),
        ("B", c_int32), ("N", c_int32), ("K", c_int32), ("T", c_int32),
        ("pitch", c_int64), ("pitch_grad", c_int64),
        ("mask_weight_masked", c_float), ("mask_weight_unmasked", c_float),
        ("backward", c_int32), ("stream", c_void_p), ("logits_dtype", c_int32),
    ]


class HeadDesc(ctypes.Structure):
    """Mirror of `d3pm_head_desc`."""
    _fields_ = [
        ("hidden_c", c_void_p), ("hidden_u", c_void_p), ("ln_weight", c_void_p), ("ln_bias", c_void_p),
        ("w_image", c_void_p), ("bias2", c_void_p), ("x_t", c_void_p), ("t", c_void_p), ("coef_table", c_void_p),
        ("x_prev", c_void_p), ("logits_out", c_void_p), ("status", c_void_p), ("redo_rows", c_void_p),
        ("redo_count", c_void_p),
        ("B", c_int32), ("N", c_int32), ("K", c_int32), ("T", c_int32), ("D", c_int32), ("mode", c_int32),
        ("ln_eps", c_float), ("guidance_scale", c_float), ("thin_factor", c_float), ("stat_slack", c_float),
        ("seed", c_uint64), ("offset", c_uint64), ("row_offset", c_int64), ("stream", c_void_p),
    ]


DEC_MAX_TAPS, DEC_MAX_CLASSES = 32, 8


class DecConvDesc(ctypes.Structure):
    """Mirror of `d3pm_dec_conv_desc`."""
    _fields_ = [
        ("x", c_void_p), ("in_scale", c_void_p), ("in_shift", c_void_p), ("w_image", c_void_p), ("bias", c_void_p),
        ("residual", c_void_p), ("out", c_void_p),
        ("B", c_int32), ("T", c_int32), ("H", c_int32), ("W", c_int32), ("Cin", c_int32),
        ("ntaps", c_int32), ("nclass", c_int32), ("cta_pair", c_int32), ("Nout", c_int32), ("out_transposed", c_int32),
        ("ldo", c_int64), ("stride_t", c_int32), ("stride_h", c_int32), ("stride_w", c_int32),
        ("relu_out", c_int32), ("terms", c_int32), ("n_tile", c_int32),
        ("tap", c_int8 * 4 * DEC_MAX_TAPS * DEC_MAX_CLASSES), ("cls", c_int8 * 4 * DEC_MAX_CLASSES),
        ("stream", c_void_p),
    ]


class AttnDesc(ctypes.Structure):
    """Mirror of `d3pm_attn_desc`."""
    _fields_ = [
        ("q", c_void_p), ("k", c_void_p), ("v", c_void_p), ("y", c_void_p),
        ("B", c_int32), ("N", c_int32), ("heads", c_int32), ("head_dim", c_int32),
        ("pitch_qkv", c_int64), ("pitch_y", c_int64), ("scale", c_float), ("stream", c_void_p),
    ]


_lib = None


def library_path() -> str:
    return os.environ.get("D3PM_B200_LIB", os.path.join(_HERE, "csrc", _LIB_NAME))


def load_library() -> ctypes.CDLL:
    """Load the shared library once; raise `D3PMError` (never fall back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.isfile(path):
        raise D3PMError(
            f"{path} not found: build it with `python __graft_entry__.py build` (or `make -C "
            f"{os.path.join(_HERE, 'csrc')}`); this package has no non-CUDA fallback")
    try:
        lib = ctypes.CDLL(path)
    except OSError as exc:  # e.g. libcudart missing
        raise D3PMError(f"cannot load {path}: {exc}") from exc
    missing = [s for s in EXPORTED_SYMBOLS if not hasattr(lib, s)]
    if missing:
        raise D3PMError(f"{path} lacks symbols {missing}; rebuild it")

    lib.d3pm_version.restype = c_int
    lib.d3pm_version.argtypes = []
    lib.d3pm_last_error.restype = c_char_p
    lib.d3pm_last_error.argtypes = []
    lib.d3pm_build_coef_table.restype = c_int
    lib.d3pm_build_coef_table.argtypes = [c_void_p, c_int, c_int, c_void_p, c_void_p]
    lib.d3pm_fused_step.restype = c_int
    lib.d3pm_fused_step.argtypes = [POINTER(StepDesc)]
    lib.d3pm_philox_uniform.restype = c_int
    lib.d3pm_philox_uniform.argtypes = [c_void_p, c_int64, c_int, c_int64, c_uint64, c_uint64, c_int64, c_void_p]
    lib.d3pm_q_posterior.restype = c_int
    lib.d3pm_q_posterior.argtypes = [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                     c_int, c_int, c_int, c_int, c_void_p, c_void_p]
    lib.d3pm_gumbel_argmax.restype = c_int
    lib.d3pm_gumbel_argmax.argtypes = [c_void_p, c_int64, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int64,
                                       c_int, c_uint64, c_uint64, c_int64, c_void_p]
    lib.d3pm_tokens_to_log_onehot.restype = c_int
    lib.d3pm_tokens_to_log_onehot.argtypes = [c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p]
    lib.d3pm_argmax_classes.restype = c_int
    lib.d3pm_argmax_classes.argtypes = [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int, c_int,
                                        c_void_p]
    lib.d3pm_q_sample_tokens.restype = c_int
    lib.d3pm_q_sample_tokens.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_uint64, c_uint64, c_int64,
                                         c_void_p, c_void_p, c_void_p]
    lib.d3pm_q_pred.restype = c_int
    lib.d3pm_q_pred.argtypes = [c_void_p, c_int64, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_int, c_int, c_int,
                                c_int, c_void_p]
    lib.d3pm_purity_select.restype = c_int
    lib.d3pm_purity_select.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                       c_int, c_uint64, c_uint64, c_int64, c_void_p]
    lib.d3pm_head_image_floats.restype = c_int64
    lib.d3pm_head_image_floats.argtypes = [c_int, c_int]
    lib.d3pm_head_prepare.restype = c_int
    lib.d3pm_head_prepare.argtypes = [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.d3pm_head_step.restype = c_int
    lib.d3pm_head_step.argtypes = [POINTER(HeadDesc)]
    lib.d3pm_decode_lut.restype = c_int
    lib.d3pm_decode_lut.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]
    lib.d3pm_tokens_to_features.restype = c_int
    lib.d3pm_tokens_to_features.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]
    lib.d3pm_scale_rows.restype = c_int
    lib.d3pm_scale_rows.argtypes = [c_void_p, c_int64, c_void_p, c_int, c_int, c_int, c_void_p]
    lib.d3pm_train_rows.restype = c_int
    lib.d3pm_train_rows.argtypes = [POINTER(TrainDesc)]
    lib.d3pm_host_step_create.restype = c_int
    lib.d3pm_host_step_create.argtypes = [POINTER(c_void_p), c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int]
    lib.d3pm_host_step_destroy.restype = c_int
    lib.d3pm_host_step_destroy.argtypes = [c_void_p]
    lib.d3pm_host_step_h2d_bytes.restype = c_int64
    lib.d3pm_host_step_h2d_bytes.argtypes = [c_void_p]
    lib.d3pm_host_step_d2h_bytes.restype = c_int64
    lib.d3pm_host_step_d2h_bytes.argtypes = [c_void_p]
    lib.d3pm_host_step_set_logits_dtype.restype = c_int
    lib.d3pm_host_step_set_logits_dtype.argtypes = [c_void_p, c_int]
    lib.d3pm_host_step_run.restype = c_int
    lib.d3pm_host_step_run.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_uint64, c_uint64,
                                       c_int64, c_void_p, POINTER(c_uint32)]
    lib.d3pm_host_head_step_run.restype = c_int
    lib.d3pm_host_head_step_run.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
                                            c_void_p, c_void_p, c_void_p, c_float, c_float, c_uint64, c_uint64, c_int64,
                                            c_void_p, POINTER(c_uint32)]
    lib.d3pm_dec_image_floats.restype = c_int64
    lib.d3pm_dec_image_floats.argtypes = [c_int, c_int, c_int, c_int]
    lib.d3pm_dec_weight_image.restype = c_int
    lib.d3pm_dec_weight_image.argtypes = [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]
    lib.d3pm_dec_conv.restype = c_int
    lib.d3pm_dec_conv.argtypes = [POINTER(DecConvDesc)]
    lib.d3pm_dec_embed_rows.restype = c_int
    lib.d3pm_dec_embed_rows.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p]
    lib.d3pm_dec_axial_attention.restype = c_int
    lib.d3pm_dec_axial_attention.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]
    lib.d3pm_dec_col2im.restype = c_int
    lib.d3pm_dec_col2im.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                    c_void_p]
    lib.d3pm_self_attention.restype = c_int
    lib.d3pm_self_attention.argtypes = [POINTER(AttnDesc)]
    lib.d3pm_to_token_major.restype = c_int
    lib.d3pm_to_token_major.argtypes = [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_void_p]
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load_library().d3pm_last_error().decode("utf-8", "replace")
        raise D3PMError(f"{what} failed (code {rc}): {msg}")
