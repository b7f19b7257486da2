"""ctypes binding of the C ABI declared in include/cryovit_b200.h.

The library is built in-tree by ``cryovit_b200.build`` (nvcc, sm_100a). There is no fallback: if the shared
object is missing or a call fails, a :class:`CryovitB200Error` is raised.
"""
from __future__ import annotations

import ctypes
from ctypes import c_char_p, c_double, c_float, c_int, c_int64, c_void_p
from pathlib import Path

import os

# CRYOVIT_B200_LIB: load another build of the same library (A/B runs of a kernel variant, tools/build_variant.py)
LIB_PATH = Path(os.environ.get("CRYOVIT_B200_LIB") or Path(__file__).resolve().parent / "lib" / "libcryovit_b200.so")


class CryovitB200Error(RuntimeError):
    """A call across the C ABI returned a non-zero code, or the CUDA library is unavailable."""


P, I64, I32, F32, F64 = c_void_p, c_int64, c_int, c_float, c_double

# name -> argtypes; every function returns int except the two diagnostics. Mirrors include/cryovit_b200.h.
SIGNATURES: dict[str, list] = {
    "cvit_preproc_patchify": [P, I32, P, I64, I64, I64, I64, P],
    "cvit_preproc_resize_f32_3ch": [P, I32, P, I64, I64, I64, P],
    "cvit_patchify_f32_3ch": [P, P, I64, I64, I64, I64, P],
    "cvit_patch_embed_gemm": [P, I64, P, P, P, I64, I64, I64, I64, I64, I64, I64, P],
    "cvit_patch_embed_gemm_fmt": [P, I64, P, P, P, I64, I64, I64, I64, I64, I64, I64, I32, P],
    "cvit_preproc_patchify_tf32": [P, I32, P, I64, I64, I64, I64, P],
    "cvit_patchify_f32_3ch_tf32": [P, P, I64, I64, I64, I64, P],
    "cvit_layernorm_f32_tf32": [P, I64, P, P, P, I64, I64, I64, F32, P],
    "cvit_assemble_special_tokens": [P, P, I64, I64, I64, I64, P],
    "cvit_layernorm_f32_bf16": [P, I64, P, P, P, I64, I64, I64, F32, P],
    "cvit_layernorm_f32_f16": [P, I64, P, P, P, I64, I64, I64, F32, P],
    "cvit_layernorm_f32_f32": [P, I64, P, P, P, I64, I64, I64, F32, P],
    "cvit_linear_bias_bf16": [P, I64, P, P, P, I64, I64, I64, I64, I32, P],
    "cvit_linear_swiglu_bf16": [P, I64, P, P, P, I64, I64, I64, I64, P],
    "cvit_linear_scale_residual_f32": [P, I64, P, P, P, P, I64, I64, I64, I64, P],
    "cvit_linear_bias_fmt": [P, I64, P, P, P, I64, I64, I64, I64, I32, I32, P],
    "cvit_linear_bias_cfirst_f16": [P, I64, P, P, P, I64, I64, I64, I64, I32, P],
    "cvit_linear_swiglu_fmt": [P, I64, P, P, P, I64, I64, I64, I64, I32, P],
    "cvit_linear_scale_residual_fmt": [P, I64, P, P, P, P, I64, I64, I64, I64, I32, P],
    "cvit_attention_fwd_bf16": [P, P, I64, I64, I64, I64, P],
    "cvit_attention_fwd_f16": [P, P, I64, I64, I64, I64, P],
    "cvit_attention_fwd_fmt": [P, P, I64, I64, I64, I64, I32, P],
    "cvit_attention_fwd_bf16_mma_sync": [P, P, I64, I64, I64, I64, P],
    "cvit_final_norm_writeout_f16": [P, P, P, P, I64, I64, I64, I64, I64, I64, I64, F32, P],
    "cvit_features_to_ndhwc_bf16": [P, P, I64, I64, P],
    "cvit_features_f32_to_ndhwc_bf16": [P, P, I64, I64, P],
    "cvit_groupnorm_ndhwc_bf16": [P, P, P, P, P, I64, I64, I64, F32, P],
    "cvit_conv3d_dilated_ndhwc": [P, P, P, P, I64, I64, I64, I64, I64, I64, I64, P],
    "cvit_conv3d_halo_ndhwc": [P, P, P, P, I64, I64, I64, I64, I64, I64, I64, P],
    "cvit_convT_1x2x2_ndhwc": [P, P, P, P, I64, I64, I64, I64, I64, P],
    "cvit_head_tail_fused": [P, P, P, P, P, P, P, P, I64, I64, I64, P],
    "cvit_head_out_conv": [P, P, P, P, P, I64, I64, I64, P],
    "cvit_seg_stats": [P, P, I64, F32, P, P],
    "cvit_conv3d_dilated_ndhwc_act": [P, P, P, P, I64, I64, I64, I64, I64, I64, I64, I32, P],
    "cvit_conv3d_halo_ndhwc_act": [P, P, P, P, I64, I64, I64, I64, I64, I64, I64, I32, P],
    "cvit_convT_1x2x2_ndhwc_act": [P, P, P, P, I64, I64, I64, I64, I64, I32, P],
    "cvit_linear_bias_bf16_nvalid": [P, I64, P, P, P, I64, I64, I64, I64, I64, P],
    "cvit_linear_bias_bf16_nvalid_aux": [P, I64, P, P, P, I64, I64, I64, I64, I64, I32, P, P],
    "cvit_linear_bias_cfirst_f16_aux": [P, I64, P, P, P, I64, I64, I64, I64, I32, P, P],
    "cvit_conv3d_dilated_ndhwc_aux": [P, P, P, P, I64, I64, I64, I64, I64, I64, I64, I32, P, P],
    "cvit_conv3d_halo_ndhwc_aux": [P, P, P, P, I64, I64, I64, I64, I64, I64, I64, I32, P, P],
    "cvit_convT_1x2x2_ndhwc_aux": [P, P, P, P, I64, I64, I64, I64, I64, I32, P, P],
    "cvit_conv3d_wpackn_ndhwc_aux": [P, P, P, P, I64, I64, I64, I64, I64, I64, I64, I32, P, P],
    "cvit_conv3d_wpack8_aux": [P, P, P, P, I64, I64, I64, I32, P, P],
    "cvit_conv3d_rows8": [P, P, P, P, I64, I64, I64, I32, P, P, P],
    "cvit_conv3d_rows8_final": [P, P, P, P, P, I64, I64, I64, P],
    "cvit_conv3d_rows8_score": [P, P, P, P, I64, I64, I64, F32, P, P, P],
    "cvit_conv3d_rows8_score_partials": [I64, I64, I64],  # returns a size, not an error code (restype set in load())
    "cvit_conv3d_rows_ndhwc": [P, P, P, P, I64, I64, I64, I64, I64, I64, I32, P, P, P],
    "cvit_gelu_fwd_bf16": [P, P, I64, P],
    "cvit_gelu_bwd_bf16": [P, P, P, I64, P],
    "cvit_gelu_bwd_colsum_bf16": [P, P, P, P, I64, I64, P],
    "cvit_gelu_bwd_colsum_unshuffle_bf16": [P, P, P, P, I64, I64, I64, I64, P],
    "cvit_dice_bwd": [P, P, P, P, F32, P, I64, P],
    "cvit_colsum_bf16": [P, P, I64, I64, P],
    "cvit_groupnorm_bwd_ndhwc_bf16": [P, P, P, P, P, P, P, I64, I64, I64, F32, P],
    "cvit_groupnorm_bwd_gelu_ndhwc_bf16": [P, P, P, P, P, P, P, I64, I64, I64, F32, P, P, I64, P],
    "cvit_pixel_unshuffle_1x2x2_bf16": [P, P, I64, I64, I64, I64, P],
    "cvit_ndhwc_to_cfirst_padded": [P, P, I64, I64, I64, I64, I64, I64, I64, I64, I64, I64, P],
    "cvit_ndhwc_to_cfirst_padded_x3": [P, P, P, P, I64, I64, I64, I64, I64, I64, I64, I64, I64, P],
    "cvit_wgrad_splitk": [P, P, P, P, I64, I64, I64, I64, I64, I64, P],
    "cvit_wgrad_narrow_ndhwc": [P, P, P, I64, I64, I64, I64, I64, I64, P],
    "cvit_wgrad_tc8_ndhwc": [P, P, P, I64, I64, I64, I64, P],
    "cvit_wgrad_tcn_ndhwc": [P, P, P, I64, I64, I64, I64, I64, I64, P],
    "cvit_adamw_f32": [P, P, P, P, I64, F32, F32, F32, F32, F32, I64, F32, P],
    "cvit_conv3d_wpack8_gelu": [P, P, P, P, I64, I64, I64, I32, P],
    "cvit_conv3d_wpack8_final": [P, P, P, P, P, I64, I64, I64, P],
    "cvit_linear_bias_cfirst_f16_gn": [P, I64, P, P, P, I64, I64, I64, I64, I32, P, I64, P],
    "cvit_linear_bias_gelu_bf16_gn": [P, I64, P, P, P, I64, I64, I64, I64, P, I64, P],
    "cvit_convT_1x2x2_ndhwc_gn": [P, P, P, P, I64, I64, I64, I64, I64, P, I64, P],
    "cvit_groupnorm_fold": [P, I64, I64, I64, I64, F64, P, P, F32, P, P, P, I64, I64, I64, I32, P, P, P],
    "cvit_conv3d_dilated_ndhwc_tab": [P, P, P, P, I64, I64, I64, I64, I64, I64, I64, P],
    "cvit_conv3d_halo_ndhwc_tab": [P, P, P, P, I64, I64, I64, I64, I64, I64, I64, P],
    "cvit_conv3d_wpackn_ndhwc": [P, P, P, P, I64, I64, I64, I64, I64, I64, I64, I32, P],
    "cvit_wgrad_mn_ndhwc": [P, P, P, I64, I64, I64, I64, I64, I64, I64, I32, P],
    "cvit_set_gemm_pair": [I32],  # returns the previous setting, not an error code (use load().cvit_set_gemm_pair)
}

_lib: ctypes.CDLL | None = None


def load() -> ctypes.CDLL:
    """dlopen the library and bind every declared symbol (raises if any is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise CryovitB200Error(
            f"{LIB_PATH} not found: build it with `python -m cryovit_b200.build` (needs nvcc); "
            "there is no CPU fallback for the CryoVIT hot path"
        )
    lib = ctypes.CDLL(str(LIB_PATH))
    lib.cvit_last_error.restype = c_char_p
    lib.cvit_last_error.argtypes = []
    lib.cvit_abi_version.restype = c_int
    lib.cvit_abi_version.argtypes = []
    lib.cvit_conv3d_halo_weight_bytes.restype = c_int64
    lib.cvit_conv3d_halo_weight_bytes.argtypes = [c_int64, c_int64]
    for fn in (lib.cvit_conv3d_wpackn_group, lib.cvit_conv3d_wpackn_weight_bytes):
        fn.restype = c_int64
        fn.argtypes = [c_int64, c_int64]
    lib.cvit_groupnorm_fold_ab_elems.restype = c_int64
    lib.cvit_groupnorm_fold_ab_elems.argtypes = [c_int64, c_int64]
    lib.cvit_conv3d_wpack_weight_bytes.restype = c_int64
    lib.cvit_conv3d_wpack_weight_bytes.argtypes = [c_int64, c_int64]
    lib.cvit_conv3d_rows8_weight_bytes.restype = c_int64
    lib.cvit_conv3d_rows8_weight_bytes.argtypes = []
    lib.cvit_conv3d_rows_weight_bytes.restype = c_int64
    lib.cvit_conv3d_rows_weight_bytes.argtypes = [c_int64]
    lib.cvit_convT_gn_partial_rows.restype = c_int64
    lib.cvit_convT_gn_partial_rows.argtypes = [c_int64, c_int64]
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = c_int
        fn.argtypes = argtypes
    lib.cvit_conv3d_rows8_score_partials.restype = c_int64
    _lib = lib
    return lib


def call(name: str, *args) -> None:
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        msg = lib.cvit_last_error()
        raise CryovitB200Error(f"{name} failed (code {rc}): {msg.decode() if msg else '?'}")
