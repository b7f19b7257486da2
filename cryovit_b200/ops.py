"""Torch-tensor front end of the C ABI: validates dtype / layout / device, then passes raw device pointers
and the current CUDA stream across ``_lib.call``. PyTorch is used for device memory and streams only.
"""
from __future__ import annotations

import torch

from . import _lib

BF16, F16, F32, U8 = torch.bfloat16, torch.float16, torch.float32, torch.uint8


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _chk(t: torch.Tensor, dtype, name: str, contiguous: bool = True) -> int:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.CryovitB200Error(f"{name}: expected a CUDA tensor (the hot path has no CPU fallback)")
    if t.dtype != dtype:
        raise _lib.CryovitB200Error(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if contiguous and not t.is_contiguous():
        raise _lib.CryovitB200Error(f"{name}: expected a contiguous tensor")
    return t.data_ptr()


def patch_grid(H: int, W: int) -> tuple[int, int, int, int]:
    """(OH, OW, ph, pw) after the reference's pad-to-16 + x14/16 resize (vit_dataset.py:100-123)."""
    H16, W16 = (H + 15) // 16 * 16, (W + 15) // 16 * 16
    OH, OW = H16 // 16 * 14, W16 // 16 * 14
    return OH, OW, OH // 14, OW // 14


def preproc_patchify(src: torch.Tensor, out: torch.Tensor) -> None:
    """src u8|f32 [D,H,W] -> out [D*Np, Kp] (one channel, Kp >= 196): bf16, or fp32 rounded to TF32 (the TF32 patch
    embedding's operand) when ``out`` is fp32."""
    D, H, W = src.shape
    is_u8 = src.dtype == U8
    name = "cvit_preproc_patchify_tf32" if out.dtype == F32 else "cvit_preproc_patchify"
    _lib.call(name, _chk(src, U8 if is_u8 else F32, "src"), int(is_u8), _chk(out, F32 if out.dtype == F32 else BF16, "out"),
              D, H, W, out.shape[1], _stream())


def preproc_resize_3ch(src: torch.Tensor, out: torch.Tensor) -> None:
    """src u8|f32 [D,H,W] -> out f32 [D,3,OH,OW]: the reference dataset's pre-processed layout (vit_dataset.py:90-123)."""
    D, H, W = src.shape
    is_u8 = src.dtype == U8
    OH, OW, _, _ = patch_grid(H, W)
    if tuple(out.shape) != (D, 3, OH, OW):
        raise _lib.CryovitB200Error(f"preproc_resize_3ch: out must be {(D, 3, OH, OW)}, got {tuple(out.shape)}")
    _lib.call("cvit_preproc_resize_f32_3ch", _chk(src, U8 if is_u8 else F32, "src"), int(is_u8), _chk(out, F32, "out"),
              D, H, W, _stream())


def patchify_f32_3ch(src: torch.Tensor, out: torch.Tensor) -> None:
    B, C, OH, OW = src.shape
    if C != 3:
        raise _lib.CryovitB200Error("patchify_f32_3ch: expected [B,3,H,W]")
    # fp32 out: TF32-rounded patch rows for the TF32 patch embedding
    name = "cvit_patchify_f32_3ch_tf32" if out.dtype == F32 else "cvit_patchify_f32_3ch"
    _lib.call(name, _chk(src, F32, "src"), _chk(out, F32 if out.dtype == F32 else BF16, "out"), B, OH, OW, out.shape[1],
              _stream())


def patch_embed_gemm(patches, w, table, x, n_slices, n_patches, tokens, first_patch_token) -> None:
    """bf16 patches x bf16 weight, or (both fp32 holding TF32 values) a TF32 GEMM."""
    N, K = w.shape
    if patches.dtype not in (BF16, F32) or w.dtype != patches.dtype:
        raise _lib.CryovitB200Error(f"patch_embed: patches and weight must both be bf16 or both fp32, got {patches.dtype} x {w.dtype}")
    _lib.call("cvit_patch_embed_gemm_fmt", _chk(patches, patches.dtype, "patches"), patches.shape[1], _chk(w, w.dtype, "w"),
              _chk(table, F32, "table"), _chk(x, F32, "x"), x.shape[-1], n_slices, n_patches, tokens,
              first_patch_token, N, K, FMT_OPERANDS_TF32 if w.dtype == F32 else 0, _stream())


def assemble_special_tokens(x: torch.Tensor, special: torch.Tensor, B: int, T: int) -> None:
    S, C = special.shape
    _lib.call("cvit_assemble_special_tokens", _chk(x, F32, "x"), _chk(special, F32, "special"), B, T, C, S, _stream())


def layernorm(x: torch.Tensor, gamma, beta, out: torch.Tensor, eps: float, tf32: bool = False) -> None:
    """x fp32 -> out bf16 | fp16 | fp32; ``tf32`` (fp32 out only) rounds the result to TF32 for a TF32 linear."""
    M, C = x.shape
    if tf32 and out.dtype != F32:
        raise _lib.CryovitB200Error(f"layernorm: TF32 rounding needs an fp32 output, got {out.dtype}")
    if out.dtype == F32:
        _lib.call("cvit_layernorm_f32_tf32" if tf32 else "cvit_layernorm_f32_f32", _chk(x, F32, "x"), x.stride(0), _chk(gamma, F32, "gamma"),
                  _chk(beta, F32, "beta"), _chk(out, F32, "out"), out.stride(0), M, C, float(eps), _stream())
        return
    name = "cvit_layernorm_f32_f16" if out.dtype == F16 else "cvit_layernorm_f32_bf16"
    _lib.call(name, _chk(x, F32, "x"), x.stride(0), _chk(gamma, F32, "gamma"),
              _chk(beta, F32, "beta"), _chk(out, out.dtype if out.dtype == F16 else BF16, "out"), out.stride(0), M, C, float(eps), _stream())


FMT_OPERANDS_F16, FMT_OUT_F16, FMT_OPERANDS_TF32, FMT_OUT_F32 = 1, 2, 4, 8  # include/cryovit_b200.h CVIT_FMT_*


def _fmt(a, w, out=None) -> int:
    """Format flags of a linear from the tensors' own dtypes: A and W share one type -- bf16 or fp16 (a tcgen05
    kind::f16 MMA takes one type for both operands), or fp32 holding TF32 values (kind::tf32). The output may be bf16,
    fp16 or, with fp32 operands, fp32; the library refuses a combination it has no kernel for."""
    if a.dtype not in (BF16, F16, F32) or w.dtype != a.dtype:
        raise _lib.CryovitB200Error(f"linear: operands must both be bf16, both fp16 or both fp32 (TF32), got {a.dtype} x {w.dtype}")
    if out is not None and (out.dtype not in (BF16, F16, F32) or (out.dtype == F32 and a.dtype != F32)):
        raise _lib.CryovitB200Error(f"linear: output must be bf16 or fp16 (or fp32 with fp32 operands), got {out.dtype}")
    fmt = {F16: FMT_OPERANDS_F16, F32: FMT_OPERANDS_TF32}.get(a.dtype, 0)
    if out is not None:
        fmt |= {F16: FMT_OUT_F16, F32: FMT_OUT_F32}.get(out.dtype, 0)
    return fmt


def linear_bias(a, w, bias, out, gelu: bool = False) -> None:
    M, K = a.shape
    N = w.shape[0]
    fmt = _fmt(a, w, out)
    _lib.call("cvit_linear_bias_fmt", _chk(a, a.dtype, "a"), a.stride(0), _chk(w, w.dtype, "w"), _chk(bias, F32, "bias"),
              _chk(out, out.dtype, "out"), out.stride(0), M, N, K, int(gelu), fmt, _stream())


def linear_bias_cfirst(at, w, bias, out, gelu=False, aux=None) -> None:
    """out bf16 [M, N] = at[K, M]^T @ w[N, K]^T + bias (+ GELU); at and w fp16, at read as an MN-major operand.
    gelu = 2 with ``aux``: out keeps the pre-activation, aux (contiguous, out's shape) receives its GELU."""
    K, M = at.shape
    N = w.shape[0]
    act, auxp = _aux(gelu, aux, out)
    if act == 2 and (aux.stride(0) != out.stride(0)):
        raise _lib.CryovitB200Error("linear_bias_cfirst: aux must have the output's row pitch")
    _lib.call("cvit_linear_bias_cfirst_f16_aux", _chk(at, F16, "at"), at.stride(0), _chk(w, F16, "w"), _chk(bias, F32, "bias"),
              _chk(out, BF16, "out"), out.stride(0), M, N, K, act, auxp, _stream())


def gn_partials_numel(rows: int, n_cols: int, cpg: int) -> int:
    """fp32 elements of the statistics buffer a GroupNorm-producer call needs for ``rows`` GEMM rows and ``n_cols`` output
    columns in groups of ``cpg``: tiles may overhang the rows by up to a 1024-row tile."""
    return (rows + 1023) // 1024 * 32 * (n_cols // cpg) * 2


def linear_bias_cfirst_gn(at, w, bias, out, partials, cpg: int) -> None:
    """linear_bias_cfirst + GELU that also writes the GroupNorm statistics of its output (see the header)."""
    K, M = at.shape
    N = w.shape[0]
    if partials.numel() < gn_partials_numel(M, N, cpg):
        raise _lib.CryovitB200Error("linear_bias_cfirst_gn: statistics buffer too small")
    _lib.call("cvit_linear_bias_cfirst_f16_gn", _chk(at, F16, "at"), at.stride(0), _chk(w, F16, "w"), _chk(bias, F32, "bias"),
              _chk(out, BF16, "out"), out.stride(0), M, N, K, 1, _chk(partials, F32, "partials"), cpg, _stream())


def linear_bias_gelu_gn(a, w, bias, out, partials, cpg: int) -> None:
    M, K = a.shape
    N = w.shape[0]
    if partials.numel() < gn_partials_numel(M, N, cpg):
        raise _lib.CryovitB200Error("linear_bias_gelu_gn: statistics buffer too small")
    _lib.call("cvit_linear_bias_gelu_bf16_gn", _chk(a, BF16, "a"), a.stride(0), _chk(w, BF16, "w"), _chk(bias, F32, "bias"),
              _chk(out, BF16, "out"), out.stride(0), M, N, K, _chk(partials, F32, "partials"), cpg, _stream())


def convT_1x2x2_gn(x, w_sub, bias4, out, partials, cpg: int) -> tuple[int, int]:
    """Transposed convolution + GELU + the statistics of what it stores. Returns (rows, columns) of the statistics as
    ``groupnorm_fold`` wants them: (voxels, 4 Cout) in the per-32-voxel layout, or (32 R, 8 cpg) when the kernel kept the group
    sums in registers and wrote R rows of 8 groups (32 channels in groups of 4)."""
    D, H, W, Cin = x.shape
    Cout = w_sub.shape[0] // 4
    R = int(_lib.load().cvit_convT_gn_partial_rows(Cout, cpg))
    if partials.numel() < max(gn_partials_numel(D * H * W, 4 * Cout, cpg), R * 16):
        raise _lib.CryovitB200Error("convT_1x2x2_gn: statistics buffer too small")
    _lib.call("cvit_convT_1x2x2_ndhwc_gn", _chk(x, BF16, "x"), _chk(w_sub, BF16, "w_sub"), _chk(bias4, F32, "bias4"),
              _chk(out, BF16, "out"), D, H, W, Cin, Cout, _chk(partials, F32, "partials"), cpg, _stream())
    return (32 * R, 8 * cpg) if R else (D * H * W, 4 * Cout)


LAYOUT_TAPS, LAYOUT_HALO, LAYOUT_WPACKN, LAYOUT_ROWS = 0, 1, 2, 3


def groupnorm_fold_ab(channels: int, groups: int, device) -> torch.Tensor:
    """The zero-filled scale / shift + scratch buffer groupnorm_fold works in (allocate once per layer)."""
    return torch.zeros(int(_lib.load().cvit_groupnorm_fold_ab_elems(channels, groups)), device=device, dtype=F32)


def groupnorm_fold(partials, rows: int, partial_cols: int, groups: int, n_per_group: int, gamma, beta, eps: float, ab,
                   w32, w_out, cin: int, cout_pad: int, layout: int, bias, table) -> None:
    """Statistics partials of ``rows`` producer rows -> scale / shift (ab) -> folded bf16 weights + 64-row bias table."""
    C = gamma.numel()
    if w_out.numel() != w32.numel() or table.numel() != 64 * cout_pad or \
            ab.numel() < _lib.load().cvit_groupnorm_fold_ab_elems(C, groups):
        raise _lib.CryovitB200Error("groupnorm_fold: buffer sizes do not match the layer")
    _lib.call("cvit_groupnorm_fold", _chk(partials, F32, "partials"), (rows + 31) // 32, partial_cols, groups, C, float(n_per_group),
              _chk(gamma, F32, "gamma"), _chk(beta, F32, "beta"), float(eps), _chk(ab, F32, "ab"), _chk(w32, F32, "w32"),
              _chk(w_out, BF16, "w_out"), w32.numel(), cin, cout_pad, layout, _chk(bias, F32, "bias"), _chk(table, F32, "table"),
              _stream())


def conv3d_dilated_tab(x, w_taps, table, out, dil: int) -> None:
    D, H, W, Cin = x.shape
    Cout = w_taps.shape[0] // 27
    _lib.call("cvit_conv3d_dilated_ndhwc_tab", _chk(x, BF16, "x"), _chk(w_taps, BF16, "w_taps"), _chk(table, F32, "table"),
              _chk(out, BF16, "out"), D, H, W, Cin, Cout, out.shape[-1], dil, _stream())


def conv3d_halo_tab(x, w_img, table, out, dil: int, cout_pad: int) -> None:
    D, H, W, Cin = x.shape
    _lib.call("cvit_conv3d_halo_ndhwc_tab", _chk(x, BF16, "x"), _chk(w_img, BF16, "w_img"), _chk(table, F32, "table"),
              _chk(out, BF16, "out"), D, H, W, Cin, cout_pad, out.shape[-1], dil, _stream())


def wpackn_group(cin: int, cout_pad: int) -> int:
    """Voxels per tensor-core row of the W-packed narrow-layer kernel for this layer; 0 = no such kernel."""
    return int(_lib.load().cvit_conv3d_wpackn_group(cin, cout_pad))


def _aux(act, aux, out):
    """(act, aux pointer) of the *_aux entry points: act 0 none, 1 GELU, 2 out = z and aux = gelu(z), 3 out = y * gelu'(aux)."""
    act = int(act)
    if act >= 2:
        if aux is None or tuple(aux.shape) != tuple(out.shape):
            raise _lib.CryovitB200Error(f"act={act} needs an aux tensor of the output's shape {tuple(out.shape)}")
        return act, _chk(aux, BF16, "aux")
    return act, None


def conv3d_wpackn(x, w_img, table, out, dil: int, cout_pad: int, act=True, aux=None) -> None:
    """Narrow-layer (Cin 16 / 32) dilated conv + bias-table row + GELU, P output voxels of a row per MMA row (csrc/conv_wpackn.cu)."""
    D, H, W, Cin = x.shape
    if w_img.numel() * 2 != _lib.load().cvit_conv3d_wpackn_weight_bytes(Cin, cout_pad):
        raise _lib.CryovitB200Error("conv3d_wpackn: weight image does not match the layer")
    act, auxp = _aux(act, aux, out)
    _lib.call("cvit_conv3d_wpackn_ndhwc_aux", _chk(x, BF16, "x"), _chk(w_img, BF16, "w_img"), _chk(table, F32, "table"),
              _chk(out, BF16, "out"), D, H, W, Cin, cout_pad, out.shape[-1], dil, act, auxp, _stream())


def linear_swiglu(a, w12i, bias12i, out) -> None:
    M, K = a.shape
    N2 = w12i.shape[0]
    fmt = _fmt(a, w12i, out)
    _lib.call("cvit_linear_swiglu_fmt", _chk(a, a.dtype, "a"), a.stride(0), _chk(w12i, w12i.dtype, "w12i"),
              _chk(bias12i, F32, "bias12i"), _chk(out, out.dtype, "out"), out.stride(0), M, N2, K, fmt, _stream())


def linear_scale_residual(a, w, bias, gamma, x) -> None:
    M, K = a.shape
    N = w.shape[0]
    fmt = _fmt(a, w)
    _lib.call("cvit_linear_scale_residual_fmt", _chk(a, a.dtype, "a"), a.stride(0), _chk(w, w.dtype, "w"),
              _chk(bias, F32, "bias"), _chk(gamma, F32, "gamma"), _chk(x, F32, "x"), x.stride(0), M, N, K, fmt, _stream())


def attention(qkv, out, n_slices: int, tokens: int, heads: int, legacy_mma_sync: bool = False) -> None:
    """out bf16 | fp16 | fp32 (TF32-rounded, from bf16 q/k/v only)."""
    if not legacy_mma_sync:
        if qkv.dtype not in (BF16, F16) or out.dtype not in (BF16, F16, F32) or (qkv.dtype == F16 and out.dtype != F16):
            raise _lib.CryovitB200Error(f"attention: unsupported formats qkv {qkv.dtype} -> out {out.dtype}")
        fmt = (FMT_OPERANDS_F16 if qkv.dtype == F16 else 0) | {F16: FMT_OUT_F16, F32: FMT_OUT_F32}.get(out.dtype, 0)
        _lib.call("cvit_attention_fwd_fmt", _chk(qkv, qkv.dtype, "qkv"), _chk(out, out.dtype, "out"), n_slices, tokens, heads, 64,
                  fmt, _stream())
        return
    _lib.call("cvit_attention_fwd_bf16_mma_sync" if legacy_mma_sync else "cvit_attention_fwd_bf16", _chk(qkv, BF16, "qkv"), _chk(out, BF16, "out"), n_slices, tokens, heads, 64,
              _stream())


def final_norm_writeout(x, gamma, beta, features, n_slices, tokens, first_patch_token, n_patches, d0, eps) -> None:
    C, D_total = features.shape[0], features.shape[1]
    _lib.call("cvit_final_norm_writeout_f16", _chk(x, F32, "x"), _chk(gamma, F32, "gamma"), _chk(beta, F32, "beta"),
              _chk(features, F16, "features"), n_slices, tokens, first_patch_token, n_patches, C, D_total, d0,
              float(eps), _stream())


# ------------------------------------------------------------------------------------------------- head
def features_to_ndhwc(features: torch.Tensor, out: torch.Tensor) -> None:
    C = features.shape[0]
    DHW = features.numel() // C
    if features.dtype == F32:
        _lib.call("cvit_features_f32_to_ndhwc_bf16", _chk(features, F32, "features"), _chk(out, BF16, "out"), C, DHW,
                  _stream())
        return
    _lib.call("cvit_features_to_ndhwc_bf16", _chk(features, F16, "features"), _chk(out, BF16, "out"), C, DHW, _stream())


def groupnorm_ndhwc(x, out, gamma, beta, stats, groups: int, eps: float) -> None:
    C = x.shape[-1]
    DHW = x.numel() // C
    _lib.call("cvit_groupnorm_ndhwc_bf16", _chk(x, BF16, "x"), _chk(out, BF16, "out"), _chk(gamma, F32, "gamma"),
              _chk(beta, F32, "beta"), _chk(stats, F32, "stats"), DHW, C, groups, float(eps), _stream())


def conv3d_dilated(x, w_taps, bias, out, dil: int) -> None:
    D, H, W, Cin = x.shape
    Cout = w_taps.shape[0] // 27
    _lib.call("cvit_conv3d_dilated_ndhwc", _chk(x, BF16, "x"), _chk(w_taps, BF16, "w_taps"), _chk(bias, F32, "bias"),
              _chk(out, BF16, "out"), D, H, W, Cin, Cout, out.shape[-1], dil, _stream())


def conv3d_halo(x, w_img, bias, out, dil: int, cout_pad: int) -> None:
    """Narrow-layer (Cin 8/16/32) dilated conv + bias + GELU from a shared-memory halo tile; see the header."""
    D, H, W, Cin = x.shape
    if w_img.numel() * 2 != _lib.load().cvit_conv3d_halo_weight_bytes(Cin, cout_pad):
        raise _lib.CryovitB200Error(f"conv3d_halo: weight image has {w_img.numel() * 2} bytes, expected "
                                    f"{_lib.load().cvit_conv3d_halo_weight_bytes(Cin, cout_pad)}")
    _lib.call("cvit_conv3d_halo_ndhwc", _chk(x, BF16, "x"), _chk(w_img, BF16, "w_img"), _chk(bias, F32, "bias"),
              _chk(out, BF16, "out"), D, H, W, Cin, cout_pad, out.shape[-1], dil, _stream())


def conv3d_wpack8_gelu(x, w_img, bias_n, out, act=True, aux=None) -> None:
    """output_layer.0 (8 -> 8, k3) + bias + GELU with 8 output voxels of a row per MMA row (csrc/conv_wpack.cu)."""
    D, H, W, Cin = x.shape
    if Cin != 8 or w_img.numel() * 2 != _lib.load().cvit_conv3d_wpack_weight_bytes(8, 8):
        raise _lib.CryovitB200Error("conv3d_wpack8_gelu: needs 8 input channels and the (P=8, Cout=8) weight image")
    act, auxp = _aux(act, aux, out)
    _lib.call("cvit_conv3d_wpack8_aux", _chk(x, BF16, "x"), _chk(w_img, BF16, "w_img"), _chk(bias_n, F32, "bias_n"),
              _chk(out, BF16, "out"), D, H, W, act, auxp, _stream())


def rows_supported(cin: int, cout: int) -> bool:
    """Is there a one-voxel-per-row kernel (csrc/conv_rows.cu) for this narrow layer?"""
    return cin in (16, 32) and cout in (16, 32)


def conv3d_rows(x, w_img, table, out, dil: int, act=True, aux=None, db=None) -> None:
    """Narrow-layer (16 / 32 channels) dilated conv + bias-table row (+ GELU), one voxel per MMA row (csrc/conv_rows.cu)."""
    D, H, W, Cin = x.shape
    Cout = out.shape[-1]
    if not rows_supported(Cin, Cout) or w_img.numel() * 2 != (Cout // 16) * _lib.load().cvit_conv3d_rows_weight_bytes(Cin) or \
            table.numel() != 64 * Cout:
        raise _lib.CryovitB200Error("conv3d_rows: weight image / bias table do not match the layer")
    act, auxp = _aux(act, aux, out)
    _lib.call("cvit_conv3d_rows_ndhwc", _chk(x, BF16, "x"), _chk(w_img, BF16, "w_img"), _chk(table, F32, "table"),
              _chk(out, BF16, "out"), D, H, W, Cin, Cout, dil, act, auxp, _chk(db, F32, "db") if db is not None else None, _stream())


def conv3d_rows8(x, w_img, bias8, out, act=True, aux=None, db=None) -> None:
    """output_layer.0 (8 -> 8, k3, dilation 1) + bias (+ GELU), one voxel per MMA row (csrc/conv_rows8.cu); W % 8 == 0."""
    D, H, W, Cin = x.shape
    if Cin != 8 or w_img.numel() * 2 != _lib.load().cvit_conv3d_rows8_weight_bytes():
        raise _lib.CryovitB200Error("conv3d_rows8: needs 8 input channels and the rows8 weight image")
    act, auxp = _aux(act, aux, out)
    _lib.call("cvit_conv3d_rows8", _chk(x, BF16, "x"), _chk(w_img, BF16, "w_img"), _chk(bias8, F32, "bias8"),
              _chk(out, BF16, "out"), D, H, W, act, auxp, _chk(db, F32, "db") if db is not None else None, _stream())


def conv3d_rows8_final(x, w_img, bias1, logits=None, probs=None) -> None:
    """output_layer.2 (8 -> 1, k3) + bias + clip(-5, 5) (+ sigmoid), one voxel per MMA row (csrc/conv_rows8.cu); W % 8 == 0."""
    D, H, W, Cin = x.shape
    if Cin != 8 or w_img.numel() * 2 != _lib.load().cvit_conv3d_rows8_weight_bytes():
        raise _lib.CryovitB200Error("conv3d_rows8_final: needs 8 input channels and the rows8 weight image")
    _lib.call("cvit_conv3d_rows8_final", _chk(x, BF16, "x"), _chk(w_img, BF16, "w_img"), _chk(bias1, F32, "bias1"),
              _chk(logits, F32, "logits") if logits is not None else None, _chk(probs, F32, "probs") if probs is not None else None,
              D, H, W, _stream())


def conv3d_rows8_score(x, w_img, bias1, labels, partials, out8, threshold: float = 0.5) -> torch.Tensor:
    """output_layer.2 (8 -> 1, k3) + bias + clip(-5, 5) + sigmoid as ``conv3d_rows8_final``, scored instead of stored: ``out8``
    (fp64 [8], overwritten) = the eight masked sums of ``seg_stats`` against int8 ``labels`` [D, H, W] (-1 = ignore).
    ``partials``: fp64 scratch of at least ``rows8_score_partials(D, H, W)`` numbers. W % 8 == 0."""
    D, H, W, Cin = x.shape
    if Cin != 8 or w_img.numel() * 2 != _lib.load().cvit_conv3d_rows8_weight_bytes():
        raise _lib.CryovitB200Error("conv3d_rows8_score: needs 8 input channels and the rows8 weight image")
    if tuple(labels.shape) != (D, H, W) or out8.numel() != 8 or partials.numel() < rows8_score_partials(D, H, W):
        raise _lib.CryovitB200Error(f"conv3d_rows8_score: labels {tuple(labels.shape)} must be {(D, H, W)}, out8 fp64 [8], "
                                    f"partials >= {rows8_score_partials(D, H, W)} doubles")
    _lib.call("cvit_conv3d_rows8_score", _chk(x, BF16, "x"), _chk(w_img, BF16, "w_img"), _chk(bias1, F32, "bias1"),
              _chk(labels, torch.int8, "labels"), D, H, W, float(threshold), _chk(partials, torch.float64, "partials"),
              _chk(out8, torch.float64, "out8"), _stream())
    return out8


def rows8_score_partials(D: int, H: int, W: int) -> int:
    """fp64 scratch numbers ``conv3d_rows8_score`` needs for a [D, H, W] volume."""
    return int(_lib.load().cvit_conv3d_rows8_score_partials(D, H, W))


def conv3d_wpack8_final(x, w_img, bias_n, logits=None, probs=None) -> None:
    """output_layer.2 (8 -> 1, k3) + bias + clip(-5, 5) (+ sigmoid) with 16 output voxels of a row per MMA row."""
    D, H, W, Cin = x.shape
    if Cin != 8 or w_img.numel() * 2 != _lib.load().cvit_conv3d_wpack_weight_bytes(16, 1):
        raise _lib.CryovitB200Error("conv3d_wpack8_final: needs 8 input channels and the (P=16, Cout=1) weight image")
    _lib.call("cvit_conv3d_wpack8_final", _chk(x, BF16, "x"), _chk(w_img, BF16, "w_img"), _chk(bias_n, F32, "bias_n"),
              _chk(logits, F32, "logits") if logits is not None else None,
              _chk(probs, F32, "probs") if probs is not None else None, D, H, W, _stream())


def convT_1x2x2(x, w_sub, bias4, out) -> None:
    D, H, W, Cin = x.shape
    Cout = w_sub.shape[0] // 4
    _lib.call("cvit_convT_1x2x2_ndhwc", _chk(x, BF16, "x"), _chk(w_sub, BF16, "w_sub"), _chk(bias4, F32, "bias4"),
              _chk(out, BF16, "out"), D, H, W, Cin, Cout, _stream())


def head_tail(x, w1, b1, w2, b2, scratch, logits=None, probs=None) -> None:
    D, H, W, _ = x.shape
    _lib.call("cvit_head_tail_fused", _chk(x, BF16, "x"), _chk(w1, F32, "w1"), _chk(b1, F32, "b1"),
              _chk(w2, F32, "w2"), _chk(b2, F32, "b2"),
              _chk(logits, F32, "logits") if logits is not None else None,
              _chk(probs, F32, "probs") if probs is not None else None, _chk(scratch, BF16, "scratch"), D, H, W,
              _stream())


def head_out_conv(x, w2, b2, logits=None, probs=None) -> None:
    D, H, W, _ = x.shape
    _lib.call("cvit_head_out_conv", _chk(x, BF16, "x"), _chk(w2, F32, "w2"), _chk(b2, F32, "b2"),
              _chk(logits, F32, "logits") if logits is not None else None,
              _chk(probs, F32, "probs") if probs is not None else None, D, H, W, _stream())


def seg_stats(probs: torch.Tensor, labels: torch.Tensor, threshold: float = 0.5) -> torch.Tensor:
    """Masked (label > -1) reductions behind DiceLoss / DiceMetric / F1Metric, fp64 [8] on the device (see the header)."""
    out = torch.zeros(8, device=probs.device, dtype=torch.float64)
    _lib.call("cvit_seg_stats", _chk(probs, F32, "probs"), _chk(labels, F32, "labels"), probs.numel(), float(threshold),
              out.data_ptr(), _stream())
    return out
