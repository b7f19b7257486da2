"""Torch-tensor front end of the TRAINING entry points of the C ABI (see include/cryovit_b200.h, "Head TRAINING")."""
from __future__ import annotations

import os

import torch

from . import _lib
from .ops import BF16, F32, _aux, _chk, _stream, det_scratch

# Every reduction below that ends in float atomics takes ``det``: None (default) keeps the atomic kernel; a scratch provider
# (ops.det_scratch) selects its deterministic variant, per-block partial rows added in a fixed order (csrc/det_reduce.cuh).


def conv3d_dilated_act(x, w_taps, bias, out, dil: int, act, aux=None) -> None:
    """act: 0 none, 1 GELU, 2 out = z and aux = gelu(z), 3 out = y * gelu'(aux) (include/cryovit_b200.h, *_aux)."""
    D, H, W, Cin = x.shape
    Cout = w_taps.shape[0] // 27
    act, auxp = _aux(act, aux, out)
    _lib.call("cvit_conv3d_dilated_ndhwc_aux", _chk(x, BF16, "x"), _chk(w_taps, BF16, "w_taps"), _chk(bias, F32, "bias"),
              _chk(out, BF16, "out"), D, H, W, Cin, Cout, out.shape[-1], dil, act, auxp, _stream())


def conv3d_halo_act(x, w_img, bias, out, dil: int, cout_pad: int, act, aux=None) -> None:
    D, H, W, Cin = x.shape
    act, auxp = _aux(act, aux, out)
    _lib.call("cvit_conv3d_halo_ndhwc_aux", _chk(x, BF16, "x"), _chk(w_img, BF16, "w_img"), _chk(bias, F32, "bias"),
              _chk(out, BF16, "out"), D, H, W, Cin, cout_pad, out.shape[-1], dil, act, auxp, _stream())


def convT_act(x, w_sub, bias4, out, act, aux=None) -> None:
    D, H, W, Cin = x.shape
    Cout = w_sub.shape[0] // 4
    act, auxp = _aux(act, aux, out)
    _lib.call("cvit_convT_1x2x2_ndhwc_aux", _chk(x, BF16, "x"), _chk(w_sub, BF16, "w_sub"), _chk(bias4, F32, "bias4"),
              _chk(out, BF16, "out"), D, H, W, Cin, Cout, act, auxp, _stream())


def linear_nvalid(a, w, bias, out, n_valid: int, z=None) -> None:
    """out[M, n_valid] = a[M, K] @ w[N, K]^T + bias (no activation); w may carry zero rows beyond n_valid. With ``z``
    (bf16, out's shape and pitch) the result is multiplied by gelu'(z): the gradient of the pre-activation z."""
    M, K = a.shape
    act, auxp = _aux(3 if z is not None else 0, z, out)
    if z is not None and z.stride(0) != out.stride(0):
        raise _lib.CryovitB200Error("linear_nvalid: z must have the output's row pitch")
    _lib.call("cvit_linear_bias_bf16_nvalid_aux", _chk(a, BF16, "a"), a.stride(0), _chk(w, BF16, "w"), _chk(bias, F32, "bias"),
              _chk(out, BF16, "out"), out.stride(0), M, w.shape[0], K, n_valid, act, auxp, _stream())


def gelu_fwd(z, a) -> None:
    _lib.call("cvit_gelu_fwd_bf16", _chk(z, BF16, "z"), _chk(a, BF16, "a"), z.numel(), _stream())


def gelu_bwd_unshuffle(da, z, dzun, db, det=None) -> None:
    """dz = da * gelu'(z) over a [D, H2, W2, C] volume, stored pixel-unshuffled into dzun [D, H2/2, W2/2, 4C]
    ((i, j, c) channel order), db += column sums of dz."""
    D, H2, W2, C = z.shape
    if tuple(dzun.shape) != (D, H2 // 2, W2 // 2, 4 * C):
        raise _lib.CryovitB200Error(f"gelu_bwd_unshuffle: dzun {tuple(dzun.shape)} does not match z {tuple(z.shape)}")
    if det is not None:
        sp, sn = det_scratch(det, "scratch", _lib.load().cvit_gelu_bwd_colsum_unshuffle_bf16_det_partials(D, H2, W2, C))
        _lib.call("cvit_gelu_bwd_colsum_unshuffle_bf16_det", _chk(da, BF16, "da"), _chk(z, BF16, "z"), _chk(dzun, BF16, "dzun"),
                  _chk(db, F32, "db"), D, H2, W2, C, sp, sn, _stream())
        return
    _lib.call("cvit_gelu_bwd_colsum_unshuffle_bf16", _chk(da, BF16, "da"), _chk(z, BF16, "z"), _chk(dzun, BF16, "dzun"),
              _chk(db, F32, "db"), D, H2, W2, C, _stream())


def gelu_bwd(da, z, dz, db=None, det=None) -> None:
    """dz = da * gelu'(z); with ``db`` (fp32 [C], zeroed by the caller) also db += column sums of dz over the last axis."""
    if db is None:
        _lib.call("cvit_gelu_bwd_bf16", _chk(da, BF16, "da"), _chk(z, BF16, "z"), _chk(dz, BF16, "dz"), z.numel(), _stream())
        return
    C = z.shape[-1]
    if det is not None:
        R = z.numel() // C
        sp, sn = det_scratch(det, "scratch", _lib.load().cvit_gelu_bwd_colsum_bf16_det_partials(R, C))
        _lib.call("cvit_gelu_bwd_colsum_bf16_det", _chk(da, BF16, "da"), _chk(z, BF16, "z"), _chk(dz, BF16, "dz"), _chk(db, F32, "db"),
                  R, C, sp, sn, _stream())
        return
    _lib.call("cvit_gelu_bwd_colsum_bf16", _chk(da, BF16, "da"), _chk(z, BF16, "z"), _chk(dz, BF16, "dz"), _chk(db, F32, "db"),
              z.numel() // C, C, _stream())


def dice_bwd(logits, probs, labels, stats8, dlogit8, scale: float = 1.0) -> None:
    _lib.call("cvit_dice_bwd", _chk(logits, F32, "logits"), _chk(probs, F32, "probs"), _chk(labels, F32, "labels"),
              _chk(stats8, torch.float64, "stats8"), float(scale), _chk(dlogit8, BF16, "dlogit8"), logits.numel(), _stream())


def colsum(x, out, det=None) -> None:
    R, C = x.numel() // x.shape[-1], x.shape[-1]
    if det is not None:
        sp, sn = det_scratch(det, "scratch", _lib.load().cvit_colsum_bf16_det_partials(R, C))
        _lib.call("cvit_colsum_bf16_det", _chk(x, BF16, "x"), _chk(out, F32, "out"), R, C, sp, sn, _stream())
        return
    _lib.call("cvit_colsum_bf16", _chk(x, BF16, "x"), _chk(out, F32, "out"), R, C, _stream())


def groupnorm_bwd(x, dy, dx, gamma, stats, dgamma, dbeta, groups: int, eps: float, det=None) -> None:
    C = x.shape[-1]
    if det is not None:
        _groupnorm_bwd_det(x, dy, dx, gamma, stats, dgamma, dbeta, groups, eps, None, None, 0, det)
        return
    _lib.call("cvit_groupnorm_bwd_ndhwc_bf16", _chk(x, BF16, "x"), _chk(dy, BF16, "dy"), _chk(dx, BF16, "dx"),
              _chk(gamma, F32, "gamma"), _chk(stats, F32, "stats"), _chk(dgamma, F32, "dgamma"), _chk(dbeta, F32, "dbeta"),
              x.numel() // C, C, groups, float(eps), _stream())


def _groupnorm_bwd_det(x, dy, dx, gamma, stats, dgamma, dbeta, groups, eps, z, db, W2, det) -> None:
    C = x.shape[-1]
    DHW = x.numel() // C
    sp, sn = det_scratch(det, "scratch", _lib.load().cvit_groupnorm_bwd_gelu_ndhwc_bf16_det_partials(DHW, C, groups))
    _lib.call("cvit_groupnorm_bwd_gelu_ndhwc_bf16_det", _chk(x, BF16, "x"), _chk(dy, BF16, "dy"), _chk(dx, BF16, "dx"),
              _chk(gamma, F32, "gamma"), _chk(stats, F32, "stats"), _chk(dgamma, F32, "dgamma"), _chk(dbeta, F32, "dbeta"),
              DHW, C, groups, float(eps), None if z is None else _chk(z, BF16, "z"), None if db is None else _chk(db, F32, "db"),
              W2, sp, sn, _stream())


def groupnorm_bwd_gelu(x, dy, dz, gamma, stats, dgamma, dbeta, groups: int, eps: float, z, db, unshuffle: bool, det=None) -> None:
    """GroupNorm backward fused with the GELU backward of the layer that produced x = gelu(z): dz = d(z), db += its column sums;
    ``unshuffle``: x is [D, H2, W2, C] and dz is written as [D, H2/2, W2/2, 4C] (sub-pixel-major channels)."""
    C = x.shape[-1]
    W2 = x.shape[2] if unshuffle else 0
    if det is not None:
        _groupnorm_bwd_det(x, dy, dz, gamma, stats, dgamma, dbeta, groups, eps, z, db, W2, det)
        return
    _lib.call("cvit_groupnorm_bwd_gelu_ndhwc_bf16", _chk(x, BF16, "x"), _chk(dy, BF16, "dy"), _chk(dz, BF16, "dz"),
              _chk(gamma, F32, "gamma"), _chk(stats, F32, "stats"), _chk(dgamma, F32, "dgamma"), _chk(dbeta, F32, "dbeta"),
              x.numel() // C, C, groups, float(eps), _chk(z, BF16, "z"), _chk(db, F32, "db"), W2, _stream())


def pixel_unshuffle(src, dst) -> None:
    D, H2, W2, C = src.shape
    _lib.call("cvit_pixel_unshuffle_1x2x2_bf16", _chk(src, BF16, "src"), _chk(dst, BF16, "dst"), D, H2 // 2, W2 // 2, C, _stream())


def padded_geometry(D: int, H: int, W: int, pd: int, ph: int, pw: int) -> tuple[int, int, int, int]:
    """(Dp, Hp, Wp, pitch) of the padded channels-first operand: Wp and the row pitch are multiples of 8."""
    Dp, Hp, Wp = D + 2 * pd, H + 2 * ph, (W + 2 * pw + 7) // 8 * 8
    return Dp, Hp, Wp, Dp * Hp * Wp


def to_cfirst_padded(x, out, pd: int, ph: int, pw: int, wshift: int = 0) -> None:
    """x bf16 [D,H,W,C] -> out bf16 [C, pitch] (channels first, zero padded, columns shifted by wshift)."""
    D, H, W, C = x.shape
    _, _, Wp, _ = padded_geometry(D, H, W, pd, ph, pw)
    _lib.call("cvit_ndhwc_to_cfirst_padded", _chk(x, BF16, "x"), _chk(out, BF16, "out"), D, H, W, C, pd, ph, pw, Wp, wshift,
              out.shape[1], _stream())


def to_cfirst_padded_x3(x, outs, pd: int, ph: int, pw: int) -> None:
    """The three column-shifted copies (-1, 0, +1) of a narrow volume (C in {8, 16, 32}) in one pass."""
    D, H, W, C = x.shape
    _, _, Wp, pitch = padded_geometry(D, H, W, pd, ph, pw)
    _lib.call("cvit_ndhwc_to_cfirst_padded_x3", _chk(x, BF16, "x"), _chk(outs[0], BF16, "out"), _chk(outs[1], BF16, "out"),
              _chk(outs[2], BF16, "out"), D, H, W, C, pd, ph, pw, Wp, pitch, _stream())


def wgrad_mn(a, b, out, dil: int = 1, shift_a: bool = False, det=None) -> None:
    """out[t, m, n] += sum_v a[v + off_a(t), m] * b[v + off_b(t), n] from channels-last bf16 volumes [D,H,W,C] (27 taps) or
    [rows, C] matrices (one tap); see cvit_wgrad_mn_ndhwc."""
    ntaps = out.shape[0]
    if a.dim() == 2:
        D, H, W = 1, 1, a.shape[0]
    else:
        D, H, W = a.shape[:3]
    if det is not None:
        sp, sn = det_scratch(det, "scratch", _lib.load().cvit_wgrad_mn_ndhwc_det_partials(D, H, W, a.shape[-1], b.shape[-1], ntaps))
        _lib.call("cvit_wgrad_mn_ndhwc_det", _chk(a, BF16, "a"), _chk(b, BF16, "b"), _chk(out, F32, "out"), D, H, W, a.shape[-1],
                  b.shape[-1], dil, ntaps, int(shift_a), sp, sn, _stream())
        return
    _lib.call("cvit_wgrad_mn_ndhwc", _chk(a, BF16, "a"), _chk(b, BF16, "b"), _chk(out, F32, "out"), D, H, W, a.shape[-1], b.shape[-1],
              dil, ntaps, int(shift_a), _stream())


def rows_weight_gradient(x_rows, dz_rows, det=None):
    """dW[M, N] = dz_rows^T @ x_rows for row-major bf16 [R, N] / [R, M] (1x1x1 and transposed convolutions) without any
    transposed copy, or None when the shapes do not fit the MN-major kernel (then the caller uses the split-K path).
    Operands narrower than 64 channels are widened by viewing f consecutive rows as one row of f x C channels (both
    operands alike): the product then holds f x f blocks of which the f diagonal ones sum to dW."""
    R, N = x_rows.shape
    M = dz_rows.shape[1]
    f = 1
    while min(M, N) * f < 64:
        f *= 2
    if R % f or (M * f) % 8 or (N * f) % 8 or not x_rows.is_contiguous() or not dz_rows.is_contiguous():
        return None
    a, b = dz_rows.view(R // f, f * M), x_rows.view(R // f, f * N)
    out = torch.zeros(1, f * M, f * N, device=x_rows.device, dtype=F32)
    wgrad_mn(a, b, out, det=det)
    if f == 1:
        return out[0]
    blocks = out[0].view(f, M, f, N)
    return sum(blocks[i, :, i, :] for i in range(f))


_KOFFS: dict = {}


def narrow_wgrad_switches_off() -> list[str]:
    """The switches set to select the atomic CUDA-core kernel (cvit_wgrad_narrow_ndhwc) for the narrow layers' weight gradients:
    a path deterministic mode has no variant of."""
    return [k for k in ("CVIT_WGRAD_TC8", "CVIT_WGRAD_TCN") if os.environ.get(k, "1") == "0"]


def conv_weight_gradient(x, dz, dil: int, pool: dict | None = None, det=None) -> torch.Tensor:
    """dW[27, Cout, Cin] (tap = (kd*3+kh)*3+kw, fp32) of a 3x3x3 depth-dilated "same" convolution from its input x and
    output gradient dz (both bf16 [D,H,W,C]): three column-shifted channels-first copies of x, one of dz, three
    9-tap split-K GEMMs. ``pool`` (a dict) recycles the operand buffers between calls."""
    D, H, W, Cin = x.shape
    Cout = dz.shape[-1]
    if (Cin, Cout) in ((8, 8), (16, 16), (32, 16), (32, 32)):  # narrow layers: reduction over the channels-last volumes
        dwn = torch.zeros(27, Cout, Cin, device=x.device, dtype=F32)
        if Cin == 8 and W % 8 == 0 and os.environ.get("CVIT_WGRAD_TC8", "1") != "0":  # tcgen05, voxels as K (csrc/wgrad_tc.cu)
            if det is not None:
                sp, sn = det_scratch(det, "scratch", _lib.load().cvit_wgrad_tc8_ndhwc_det_partials(D, H, W))
                _lib.call("cvit_wgrad_tc8_ndhwc_det", _chk(x, BF16, "x"), _chk(dz, BF16, "dz"), _chk(dwn, F32, "dw"), D, H, W, dil,
                          sp, sn, _stream())
                return dwn
            _lib.call("cvit_wgrad_tc8_ndhwc", _chk(x, BF16, "x"), _chk(dz, BF16, "dz"), _chk(dwn, F32, "dw"), D, H, W, dil, _stream())
            return dwn
        if Cin > 8 and os.environ.get("CVIT_WGRAD_TCN", "1") != "0":
            if det is not None:
                sp, sn = det_scratch(det, "scratch", _lib.load().cvit_wgrad_tcn_ndhwc_det_partials(D, H, W, Cin, Cout))
                _lib.call("cvit_wgrad_tcn_ndhwc_det", _chk(x, BF16, "x"), _chk(dz, BF16, "dz"), _chk(dwn, F32, "dw"), D, H, W, Cin,
                          Cout, dil, sp, sn, _stream())
                return dwn
            _lib.call("cvit_wgrad_tcn_ndhwc", _chk(x, BF16, "x"), _chk(dz, BF16, "dz"), _chk(dwn, F32, "dw"), D, H, W, Cin, Cout,
                      dil, _stream())
            return dwn
        if det is not None:
            raise _lib.CryovitB200Error(
                f"deterministic mode: the {Cin} -> {Cout} weight gradient would take the atomic cvit_wgrad_narrow_ndhwc kernel "
                f"({', '.join(narrow_wgrad_switches_off()) or 'W % 8 != 0'}=0); unset the switch or turn deterministic mode off")
        _lib.call("cvit_wgrad_narrow_ndhwc", _chk(x, BF16, "x"), _chk(dz, BF16, "dz"), _chk(dwn, F32, "dw"), D, H, W, Cin, Cout,
                  dil, _stream())
        return dwn
    # Wide layers: both operands straight from the channels-last volumes (MN-major tensor-core operands, the tap is the TMA
    # box origin of the shifted one; csrc/wgrad_mn.cu). The GEMM's M is tiled in 128 channels, its N in 64 .. 256: the
    # operand whose channel count fills 128-row tiles best becomes A (1024 -> 192: x; 192 as M would waste a quarter).
    if Cin >= 64 and Cout >= 64 and Cin % 8 == 0 and Cout % 8 == 0:
        waste = lambda c: (c + 127) // 128 * 128 / c
        if waste(Cin) <= waste(Cout):
            out = torch.zeros(27, Cin, Cout, device=x.device, dtype=F32)
            wgrad_mn(x, dz, out, dil, shift_a=True, det=det)   # out[t, ci, co] = sum_v x[v + off_t, ci] dz[v, co]
            return out.transpose(1, 2)
        out = torch.zeros(27, Cout, Cin, device=x.device, dtype=F32)
        wgrad_mn(dz, x, out, dil, shift_a=False, det=det)
        return out
    # Remaining shapes: channels-first zero-padded operand copies + the K-major split-K GEMM (csrc/wgrad.cu).
    # No depth padding: a depth tap that leaves the volume shifts the K index outside [0, K), where the GEMM's TMA loads
    # read zeros anyway; only the in-plane wrap-around needs the one-voxel zero border (of dz). With the head's
    # dilations (up to 32 planes of 128) padded planes would be a third of K.
    pd = 0
    Dp, Hp, Wp, pitch = padded_geometry(D, H, W, pd, 1, 1)
    dev = x.device
    pool = pool if pool is not None else {}

    def buf(name, n):
        b = pool.get(name)
        if b is None or b.numel() < n:
            b = torch.empty(n, device=dev, dtype=BF16)
            pool[name] = b
        return b

    dzt = buf("dzt", Cout * pitch)[:Cout * pitch].view(Cout, pitch)
    to_cfirst_padded(dz, dzt, pd, 1, 1, 0)
    key = (dil, Hp, Wp, str(dev))
    if key not in _KOFFS:
        _KOFFS[key] = torch.tensor([((kd - 1) * dil * Hp + (kh - 1)) * Wp for kd in range(3) for kh in range(3)], dtype=torch.int32, device=dev)
    koffs = _KOFFS[key]
    dw = torch.zeros(3, 9, Cout, Cin, device=dev, dtype=F32)
    if Cin in (8, 16, 32):  # all three shifted copies from one pass over x
        xts = [buf(f"xt{kw}", Cin * pitch)[:Cin * pitch].view(Cin, pitch) for kw in range(3)]
        to_cfirst_padded_x3(x, xts, pd, 1, 1)
        for kw in range(3):
            wgrad_splitk(dzt, xts[kw], dw[kw], koffs, pitch, det=det)
    else:
        xt = buf("xt0", Cin * pitch)[:Cin * pitch].view(Cin, pitch)
        for kw in range(3):
            to_cfirst_padded(x, xt, pd, 1, 1, kw - 1)
            wgrad_splitk(dzt, xt, dw[kw], koffs, pitch, det=det)
    return dw.permute(1, 0, 2, 3).reshape(27, Cout, Cin)


def wgrad_splitk(at, bt, out, koffs, k: int, det=None) -> None:
    """out[t, m, n] += sum_k at[m, k] * bt[n, k + koffs[t]]; at [M, pitch], bt [N, pitch] bf16, out fp32 [T, M, N]."""
    T, M, N = out.shape
    if det is not None:
        sp, sn = det_scratch(det, "scratch", _lib.load().cvit_wgrad_splitk_det_partials(M, N, k, T))
        _lib.call("cvit_wgrad_splitk_det", _chk(at, BF16, "at"), _chk(bt, BF16, "bt"), _chk(out, F32, "out"),
                  _chk(koffs, torch.int32, "koffs"), M, N, k, at.shape[1], bt.shape[1], T, sp, sn, _stream())
        return
    _lib.call("cvit_wgrad_splitk", _chk(at, BF16, "at"), _chk(bt, BF16, "bt"), _chk(out, F32, "out"),
              _chk(koffs, torch.int32, "koffs"), M, N, k, at.shape[1], bt.shape[1], T, _stream())


def adamw(p, g, m, v, lr: float, beta1: float, beta2: float, eps: float, weight_decay: float, step: int, grad_scale: float = 1.0) -> None:
    _lib.call("cvit_adamw_f32", _chk(p, F32, "p"), _chk(g, F32, "g"), _chk(m, F32, "m"), _chk(v, F32, "v"), p.numel(),
              float(lr), float(beta1), float(beta2), float(eps), float(weight_decay), int(step), float(grad_scale), _stream())


def accumulate(dst, src) -> None:
    """dst += src over two fp32 tensors of the same size (a batch step's per-sample gradient bucket into the step's)."""
    if src.numel() != dst.numel():
        raise _lib.CryovitB200Error(f"accumulate: {src.numel()} elements into {dst.numel()}")
    _lib.call("cvit_accumulate_f32", _chk(dst, F32, "dst"), _chk(src, F32, "src"), dst.numel(), _stream())
