"""CryoVIT head TRAINING on B200 (BASELINE config 5; reference models/cryovit.py:10-83, models/base_model.py:58-63,
91-164, models/losses.py:17-32, configs/trainer/fit.yaml: AdamW lr 1e-4 / wd 1e-3, masked DiceLoss, batch of one
tomogram crop per GPU, 16-mixed precision).

One training step = forward with kept pre-activations -> masked Dice loss -> backward -> (data parallel) all-reduce of
ONE flat fp32 gradient bucket over NCCL -> fused AdamW on fp32 master weights. All arithmetic of the step runs in the
sm_100a kernels behind the C ABI:

  forward    the inference convolution kernels with act = 0 (they store the pre-activation z) + cvit_gelu_fwd
  dX         the SAME convolution kernels run on spatially flipped, channel-transposed weights (a "same" stride-1
             convolution's input gradient is a "same" convolution), act = 0, zero bias
  dW         cvit_wgrad_splitk: split-K tcgen05 GEMMs over channels-first zero-padded copies of (dZ, X)
  the rest   GELU / GroupNorm / Dice backward, pixel un-shuffle, bias column sums, AdamW (csrc/train_elementwise.cu)

torch is used for buffers, for re-packing the bf16 operand copies of the fp32 master weights each step (permutes and
casts of 8.4 M numbers) and for the NCCL all-reduce (torch.distributed): plumbing, not arithmetic of the model.
Activation gradients are bf16 (fp32 accumulation inside every kernel), weight gradients and optimizer state fp32.
"""
from __future__ import annotations

import torch

from . import nvtx, ops
from . import train_ops as T
from ._lib import CryovitB200Error
from .operand_gather import OperandGather
from .head import BLOCKS, rows8_weight_image, rowsn_weight_image, state_dict_keys, wpack_weight_image, wpackn_weight_image

BF16, F32 = torch.bfloat16, torch.float32


def _taps(w: torch.Tensor, cout_pad: int) -> torch.Tensor:
    """Conv3d weight [Cout, Cin, 3,3,3] -> [27 * cout_pad, Cin] (tap-major), on the tensor's device."""
    cout, cin = w.shape[:2]
    out = torch.zeros(27, cout_pad, cin, device=w.device, dtype=w.dtype)
    out[:, :cout] = w.permute(2, 3, 4, 0, 1).reshape(27, cout, cin)
    return out.reshape(27 * cout_pad, cin)


def _halo_image(w: torch.Tensor, cout_pad: int) -> torch.Tensor:
    """cryovit_b200.head.halo_weight_image on the tensor's own device."""
    cout, cin = w.shape[:2]
    steps = cin // 16
    n_mma = 3 * steps if cin >= 16 else 2
    img = torch.zeros(9, n_mma, 2, cout_pad, 8, device=w.device, dtype=w.dtype)
    wt = w.permute(2, 3, 4, 0, 1).reshape(9, 3, cout, cin)
    if cin >= 16:
        for i in range(n_mma):
            kw, c2 = divmod(i, steps)
            for k in range(2):
                img[:, i, k, :cout] = wt[:, kw, :, c2 * 16 + k * 8: c2 * 16 + k * 8 + 8]
    else:
        img[:, 0, 0, :cout] = wt[:, 0]
        img[:, 0, 1, :cout] = wt[:, 1]
        img[:, 1, 1, :cout] = wt[:, 2]
    return img.reshape(-1)


def allreduce_gradient_bucket(flat_g: torch.Tensor) -> None:
    """Data-parallel gradient exchange: ONE all-reduce (sum) of the flat fp32 bucket holding every parameter gradient
    (8.4 M numbers, 33.6 MB: latency-bound on NVLink 5, so a single bucket rather than per-layer pieces). The 1/world
    factor is applied upstream, to the loss gradient. No-op without an initialised process group."""
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(flat_g, op=dist.ReduceOp.SUM)


class _Conv:
    """A 3x3x3 depth-dilated convolution in both directions. Narrow inputs (8/16/32 channels) use the halo kernel, the
    8 -> 8 full-resolution case the W-packed kernel. The bf16 operand images come from the trainer's per-step gather
    (``CryoVITHeadTrainerB200._pk``): ``key`` names the parameter, ``pre`` an optional re-arrangement applied first."""

    def __init__(self, trainer, key: str, cin: int, cout: int, dil: int, pre=None):
        self.tr, self.key, self.cin, self.cout, self.dil, self.pre = trainer, key, cin, cout, dil, pre

    def run(self, tag, x, wfn, bias, out, cin, cout, dil, act=0, aux=None, db=None):
        """wfn: fp32 parameter -> the [cout, cin, 3,3,3] weight of THIS convolution (identity, or flip + transpose).
        act / aux: the fused element-wise pass of the epilogue (2: out = z, aux = gelu(z); 3: out = y * gelu'(aux))."""
        if cin == 8 and cout == 8 and dil == 1 and x.shape[2] % 8 == 0 and self.tr.rows8:
            # the full-resolution 8-channel layers (output_layer.0 forward, both input gradients there): one voxel per MMA row,
            # partial sums meeting in tensor memory (csrc/conv_rows8.cu)
            b = bias.contiguous() if bias is not None else torch.zeros(8, device=x.device, dtype=F32)
            op = self.tr._pk(f"{self.key}/{tag}/rows8", self.key, lambda w: rows8_weight_image(wfn(w)))
            if act == 2 and not self.tr.fuse_store_bound:
                ops.conv3d_rows8(x, op, b, out, act=0)
                T.gelu_fwd(out, aux)
            else:
                ops.conv3d_rows8(x, op, b, out, act=act, aux=aux, db=db)
            return
        if cin == 8 and cout == 8 and dil == 1 and x.shape[2] % 16 == 0:
            # the full-resolution 8-channel layers (output_layer.0 forward, both input gradients there): W-packed kernel
            b = bias.repeat(8).contiguous() if bias is not None else torch.zeros(64, device=x.device, dtype=F32)
            op = self.tr._pk(f"{self.key}/{tag}/wpack", self.key, lambda w: wpack_weight_image(wfn(w), 8))
            if act == 2 and not self.tr.fuse_store_bound:
                # measured (profiles/r02_train_notes.md): this kernel is bound by its stores; the second store costs what
                # the separate pass does
                ops.conv3d_wpack8_gelu(x, op, b, out, act=0)
                T.gelu_fwd(out, aux)
            else:
                ops.conv3d_wpack8_gelu(x, op, b, out, act=act, aux=aux)
            return
        if ops.rows_supported(cin, cout) and self.tr.rowsn:
            # 16- / 32-channel layers (forward and input gradients alike): one voxel per tensor-core row (csrc/conv_rows.cu)
            b = bias if bias is not None else torch.zeros(cout, device=x.device, dtype=F32)
            op = self.tr._pk(f"{self.key}/{tag}/rowsn", self.key, lambda w: rowsn_weight_image(wfn(w)))
            ops.conv3d_rows(x, op, b.repeat(64).contiguous(), out, dil, act=act, aux=aux, db=db)
            return
        halo = cin in (8, 16, 32)
        cp = (32 if cout > 16 else 16) if halo else max(32, cout)
        b = torch.zeros(cp, device=x.device, dtype=F32)
        if bias is not None:
            b[:cout] = bias
        P = ops.wpackn_group(cin, cp) if halo and x.shape[2] % 4 == 0 else 0
        if P:
            # 16- / 32-channel layers (forward and input gradients alike): P voxels per tensor-core row (csrc/conv_wpackn.cu)
            op = self.tr._pk(f"{self.key}/{tag}/wpackn", self.key, lambda w: wpackn_weight_image(wfn(w), cp, P))
            ops.conv3d_wpackn(x, op, b.repeat(64), out, dil, cp, act=act, aux=aux)
        elif halo:
            op = self.tr._pk(f"{self.key}/{tag}/halo", self.key, lambda w: _halo_image(wfn(w), cp))
            T.conv3d_halo_act(x, op, b, out, dil, cp, act, aux)
        else:
            op = self.tr._pk(f"{self.key}/{tag}/taps", self.key, lambda w: _taps(wfn(w), cp))
            T.conv3d_dilated_act(x, op, b, out, dil, act, aux)

    def _w(self, w):
        return self.pre(w) if self.pre is not None else w

    def forward(self, x, bias, z, a=None):
        """z = conv(x) + bias; with ``a`` also a = gelu(z) from the same epilogue."""
        self.run("f", x, self._w, bias, z, self.cin, self.cout, self.dil, 2 if a is not None else 0, a)

    def fuses_gelu_grad(self, dz) -> bool:
        """Does the input-gradient kernel of this layer apply gelu'(z) and sum the bias gradient itself (the one-voxel-per-row
        kernels: z is prefetched before the accumulator wait)?"""
        if self.cin == 8 and self.cout == 8:
            return self.dil == 1 and dz.shape[2] % 8 == 0 and self.tr.rows8
        return ops.rows_supported(self.cout, self.cin) and self.tr.rowsn

    def input_gradient(self, dz, dx, z_below=None, db=None):
        """dx = conv^T(dz); with ``z_below`` (the pre-activation whose GELU produced this convolution's input) the
        epilogue multiplies by gelu'(z_below): dx is then the gradient of that pre-activation, and ``db`` (fp32, zeroed;
        only with ``fuses_gelu_grad``) receives its column sums."""
        # [cin, cout, 3,3,3]: the gradient convolution's weight
        self.run("g", dz, lambda w: self._w(w).flip(2, 3, 4).transpose(0, 1).contiguous(), None, dx, self.cout, self.cin, self.dil,
                 3 if z_below is not None else 0, z_below, db)


class _KeepAlivePool(dict):
    """Scratch-buffer table whose superseded entries are never freed: a captured CUDA graph has the raw pointers of
    the buffers it was captured with baked in, so a buffer that is re-allocated for a larger crop shape must stay
    alive for as long as the trainer does (otherwise a later replay of the older graph writes into memory the caching
    allocator has handed to somebody else)."""

    def __init__(self, retired: list):
        super().__init__()
        self._retired = retired

    def __setitem__(self, key, value):
        old = self.get(key)
        if old is not None and old is not value:
            self._retired.append(old)
        super().__setitem__(key, value)


class CryoVITHeadTrainerB200:
    """Data-parallel trainer of the CryoVIT head: one process per GPU, one tomogram crop per process and step."""

    def __init__(self, in_channels: int = 1536, lr: float = 1e-4, weight_decay: float = 1e-3, betas=(0.9, 0.999),
                 eps: float = 1e-8, state_dict: dict | None = None, device=None, seed: int = 0):
        if not torch.cuda.is_available():
            raise CryovitB200Error("no CUDA device: the B200 training path has no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        self.in_channels, self.lr, self.weight_decay, self.betas, self.eps = in_channels, lr, weight_decay, betas, eps
        import os

        # GELU forward (z and gelu(z) from one epilogue) and backward (gelu'(z) applied by the input-gradient epilogue)
        # fused into the convolutions; CVIT_TRAIN_FUSE_ACT=0 keeps the separate element-wise kernels (A/B, tests)
        self.fuse_activations = os.environ.get("CVIT_TRAIN_FUSE_ACT", "1") != "0"
        # ... also in the two kernels that are bound by their stores (transposed convolution, 8 -> 8 at full resolution): a loss
        # with the transposing epilogues (profiles/r02_train_notes.md), a small win since both store straight from the
        # accumulator row (19.58 -> 19.41 ms). gelu' in the input-gradient epilogues: slower than the separate pass, off.
        self.fuse_store_bound = os.environ.get("CVIT_TRAIN_FUSE_STORE_BOUND", "1") != "0"
        self.fuse_backward = os.environ.get("CVIT_TRAIN_FUSE_BWD", "0") != "0"
        self.fuse_gn_gelu = os.environ.get("CVIT_TRAIN_FUSE_GN_GELU", "1") != "0"  # GELU backward inside the GroupNorm backward pass
        # ... and inside the rows kernels' drains (z prefetched before the accumulator wait, bias gradient in registers): correct,
        # measured SLOWER in the step (19.69 vs 19.22 ms: the 8 -> 8 drain grows by 0.27 ms for a 0.39 ms pass saved, but the
        # MMAs it used to hide behind no longer cover it), off by default (profiles/r02_train_notes.md)
        self.fuse_dgrad_gelu = os.environ.get("CVIT_TRAIN_FUSE_DGRAD_GELU", "0") != "0"
        self.rows8 = os.environ.get("CVIT_HEAD_ROWS8", "1") != "0"  # 8-channel full-resolution convolutions on conv_rows8.cu
        self.rowsn = os.environ.get("CVIT_HEAD_ROWSN", "1") != "0"  # 16 / 32-channel convolutions on conv_rows.cu
        if state_dict is None:
            from .host.models import default_state_dict

            state_dict = default_state_dict(in_channels, seed=seed)  # same on every rank (fit_head passes cfg.random_seed)
        self.keys = state_dict_keys()
        sizes = [state_dict[k].numel() for k in self.keys]
        n = sum(sizes)
        self._flat_store = torch.zeros(n + 1, device=self.device, dtype=F32)  # [n] is the zero every padded operand entry reads
        self.flat_p = self._flat_store[:n]  # fp32 master weights, ONE bucket
        self.flat_g = torch.zeros(n, device=self.device, dtype=F32)  # gradients, all-reduced as one flat bucket
        self.flat_m = torch.zeros(n, device=self.device, dtype=F32)
        self.flat_v = torch.zeros(n, device=self.device, dtype=F32)
        self.p, self.g, self._offsets = {}, {}, {}
        off = 0
        for k, sz in zip(self.keys, sizes):
            shape = state_dict[k].shape
            self.p[k] = self.flat_p[off:off + sz].view(shape)
            self.g[k] = self.flat_g[off:off + sz].view(shape)
            self.p[k].copy_(state_dict[k].to(self.device, F32))
            self._offsets[k] = off
            off += sz
        self.step_count = 0
        self.launches = 0
        self._retired: list = []  # superseded scratch buffers, kept alive for the graphs captured over them
        self._gather = OperandGather(self._flat_store, self._retired)  # bf16 operand images of the weights (_pk)
        self._bufs: dict = _KeepAlivePool(self._retired)
        self._bufs["wgrad_pool"] = _KeepAlivePool(self._retired)
        self._graphs: dict = {}
        self._graph_broken = False

    # ------------------------------------------------------------------ bf16 operand images of the updated weights
    def _pk(self, name: str, key: str, fn) -> torch.Tensor:
        """The bf16 operand ``fn(p[key])`` where fn is a pure re-arrangement with zero padding (tap-major layout,
        shared-memory images, flips / transposes for input gradients ...). The weights change every step and the
        re-arrangements are dozens of small torch kernels per layer, so on first use fn runs on the parameter's GLOBAL
        INDICES (exact in fp32 up to 2^24) and the result is kept as a gather table; from the next step on ONE
        ``index_select`` over the flat bucket plus one cast produce every operand of the step (``_pk_refresh``,
        :class:`~cryovit_b200.operand_gather.OperandGather`)."""
        v = self._gather.views.get(name)
        if v is not None:
            return v
        w = self.p[key]
        if name not in self._gather.tables:
            self._gather.add(name, fn(self._gather.indices(self._offsets[key], w.shape)), BF16)
        return fn(w).to(BF16).contiguous()

    def _pk_refresh(self) -> None:
        """One gather + one cast for all operand images whose tables exist (called at the start of a step)."""
        self._gather.refresh()

    def parameter_bucket(self) -> tuple[torch.Tensor, dict[str, int], dict[str, tuple]]:
        """(fp32 [n + 1] bucket: the master weights and a trailing zero, offset and shape of every parameter): what
        ``CryoVITHeadB200.attach_bucket`` gathers its operands from."""
        return self._flat_store, dict(self._offsets), {k: tuple(v.shape) for k, v in self.p.items()}

    # ------------------------------------------------------------------ helpers
    def state_dict(self) -> dict[str, torch.Tensor]:
        return {k: v.detach().clone().cpu() for k, v in self.p.items()}

    def _buf(self, name: str, shape, dtype=BF16) -> torch.Tensor:
        n = 1
        for s in shape:
            n *= s
        b = self._bufs.get(name)
        if b is None or b.numel() < n or b.dtype != dtype:
            b = torch.empty(n, device=self.device, dtype=dtype)
            self._bufs[name] = b
        return b[:n].view(shape)

    def _gelu_bwd_bias(self, da, z, dz, key_b):
        """dz = da * gelu'(z) and the layer's bias gradient (the column sums of dz) in the same pass."""
        db = torch.zeros(z.shape[-1], device=self.device, dtype=F32)
        T.gelu_bwd(da, z, dz, db)
        self.g[key_b].copy_(db)

    def _dgrad_gelu(self, conv, dz, z_below, dz_out, key_b, tmp_name):
        """dz_out = conv^T(dz) * gelu'(z_below) (the gradient of the pre-activation below ``conv``) and that layer's bias
        gradient: inside the input-gradient kernel where it prefetches z (csrc/conv_rows*.cu), else as a second pass."""
        if self.fuse_dgrad_gelu and conv.fuses_gelu_grad(dz):
            db = torch.zeros(z_below.shape[-1], device=self.device, dtype=F32)
            conv.input_gradient(dz, dz_out, z_below=z_below, db=db)
            self.g[key_b].copy_(db)
        else:
            da = self._buf(tmp_name, tuple(dz_out.shape))
            conv.input_gradient(dz, da)
            self._gelu_bwd_bias(da, z_below, dz_out, key_b)

    def _bias_grad(self, dz, key_b):
        """The bias gradient alone (column sums of dz), for layers whose gelu' was applied by the producing epilogue."""
        db = torch.zeros(dz.shape[-1], device=self.device, dtype=F32)
        T.colsum(dz, db)
        self.g[key_b].copy_(db)

    def _wgrad_conv(self, x, dz, dil, key_w):
        """Accumulates the weight gradient of a 3x3x3 convolution into the flat bucket (the bias gradient comes out of
        ``_gelu_bwd_bias``, which produced dz)."""
        cin, cout = x.shape[-1], dz.shape[-1]
        dw = T.conv_weight_gradient(x, dz, dil, self._bufs.setdefault("wgrad_pool", {}))  # [27, cout, cin]
        self.g[key_w].copy_(dw.reshape(3, 3, 3, cout, cin).permute(3, 4, 0, 1, 2))
        self.launches += 7

    def _wgrad_rows(self, x_rows, dz_rows, xt=None):
        """dW[M, N] = dz_rows^T @ x_rows for row-major bf16 [R, N] / [R, M] (1x1x1 and transposed convolutions). ``xt``:
        x already channels-first, bf16 [N, R] with R a multiple of 8 (then x_rows is not read)."""
        if xt is None:  # straight from the row-major operands when the MN-major kernel takes the shapes (no transposed copies)
            direct = T.rows_weight_gradient(x_rows, dz_rows)
            if direct is not None:
                self.launches += 1
                return direct
        R, M = dz_rows.shape
        pitch = (R + 7) // 8 * 8
        dzt = self._buf("rows_dzt", (M, pitch))
        if xt is None:
            N = x_rows.shape[1]
            xt = self._buf("rows_xt", (N, pitch))
            T.to_cfirst_padded(x_rows.view(1, 1, R, N), xt, 0, 0, 0)  # rows along the innermost (W) axis: pitch = roundup8(R)
        else:
            N = xt.shape[0]
        T.to_cfirst_padded(dz_rows.view(1, 1, R, M), dzt, 0, 0, 0)
        dw = torch.zeros(1, M, N, device=self.device, dtype=F32)
        T.wgrad_splitk(dzt, xt, dw, torch.zeros(1, dtype=torch.int32, device=self.device), pitch)
        self.launches += 3
        return dw[0]

    # ------------------------------------------------------------------ one step
    def forward_backward(self, features: torch.Tensor, labels: torch.Tensor, grad_scale: float = 1.0) -> torch.Tensor:
        """features (C, D, h, w) fp16|fp32, labels (D, 16h, 16w) with -1 = ignore. Fills the gradient bucket and
        returns the Dice loss (0-dim tensor on the device)."""
        p, g, dev = self.p, self.g, self.device
        C, D, h, w = features.shape
        if C != self.in_channels or tuple(labels.shape) != (D, 16 * h, 16 * w):
            raise CryovitB200Error(f"features {tuple(features.shape)} / labels {tuple(labels.shape)} do not match")
        vox = D * h * w
        # CVIT_TRAIN_FUSE_ACT=0: GELU forward / backward as separate element-wise kernels (the A/B arm; default: fused
        # into the epilogues of the convolutions that produce z / the input gradients)
        fuse = self.fuse_activations
        fuse_sb, fuse_bwd = fuse and self.fuse_store_bound, fuse and self.fuse_backward
        self._pk_refresh()
        # ---------------- forward, keeping what the backward needs
        z_proj, a_proj = self._buf("z_proj", (vox, 1024)), self._buf("a_proj", (D, h, w, 1024))
        feats = features.to(dev).contiguous()
        # fp16 feature volumes whose row pitch TMA accepts: the (C, vox) layout is the projection's A operand as it lies
        # (MN-major) and, cast to bf16, already the channels-first operand of its weight gradient -- no transposes
        cfirst = feats.dtype == torch.float16 and vox % 8 == 0 and C % 8 == 0 and C >= 64
        x0 = None
        if cfirst:
            w16 = p["layers.0.weight"].reshape(1024, C).clamp(-6.0e4, 6.0e4).to(torch.float16)
            ops.linear_bias_cfirst(feats.view(C, vox), w16, p["layers.0.bias"], z_proj, gelu=2 if fuse else 0,
                                   aux=a_proj.view(vox, 1024) if fuse else None)
        else:
            x0 = self._buf("x0", (D, h, w, C))
            ops.features_to_ndhwc(feats, x0)
            ops.linear_bias(x0.view(vox, C), self._pk("proj/f", "layers.0.weight", lambda w_: w_.reshape(1024, C)), p["layers.0.bias"],
                            z_proj, gelu=False)
        if not (fuse and cfirst):
            T.gelu_fwd(z_proj, a_proj.view(vox, 1024))
        self.launches += 3
        saved = []
        cur, H, W = a_proj, h, w
        for bi, (c1, c2, c3, d1, d2) in enumerate(BLOCKS):
            pre = f"layers.{bi + 2}.layers."
            G = max(8, c1 // 8)
            n_out = self._buf(f"gn{bi}", (D, H, W, c1))
            stats = self._buf(f"gn{bi}_stats", (2 * G,), F32)
            ops.groupnorm_ndhwc(cur, n_out, p[pre + "0.weight"], p[pre + "0.bias"], stats, G, 1e-3)
            ca, cb = _Conv(self, pre + "1.weight", c1, c2, d1), _Conv(self, pre + "3.weight", c2, c2, d2)
            za, aa = self._buf(f"za{bi}", (D, H, W, c2)), self._buf(f"aa{bi}", (D, H, W, c2))
            if fuse:
                ca.forward(n_out, p[pre + "1.bias"], za, aa)
            else:
                ca.forward(n_out, p[pre + "1.bias"], za)
                T.gelu_fwd(za, aa)
            zb, ab = self._buf(f"zb{bi}", (D, H, W, c2)), self._buf(f"ab{bi}", (D, H, W, c2))
            if fuse:
                cb.forward(aa, p[pre + "3.bias"], zb, ab)
            else:
                cb.forward(aa, p[pre + "3.bias"], zb)
                T.gelu_fwd(zb, ab)
            zt, at = self._buf(f"zt{bi}", (D, 2 * H, 2 * W, c3)), self._buf(f"at{bi}", (D, 2 * H, 2 * W, c3))
            # ConvTranspose weight [c2, c3, 1, 2, 2] -> rows (i*2+j)*c3 + co of the sub-pixel GEMM
            T.convT_act(ab, self._pk(pre + "5/f", pre + "5.weight",
                                     lambda wT, c2_=c2, c3_=c3: wT[:, :, 0].permute(2, 3, 1, 0).reshape(4 * c3_, c2_)),
                        p[pre + "5.bias"].repeat(4).contiguous(), zt, 2 if fuse_sb else 0, at if fuse_sb else None)
            if not fuse_sb:
                T.gelu_fwd(zt, at)
            self.launches += 9
            saved.append((cur, n_out, stats, G, ca, za, aa, cb, zb, ab, zt, at, H, W))
            cur, H, W = at, 2 * H, 2 * W
        co = _Conv(self, "output_layer.0.weight", 8, 8, 1)
        z1, a1 = self._buf("z_o0", (D, H, W, 8)), self._buf("a_o0", (D, H, W, 8))
        if fuse:
            co.forward(cur, p["output_layer.0.bias"], z1, a1)
        else:
            co.forward(cur, p["output_layer.0.bias"], z1)
            T.gelu_fwd(z1, a1)
        logits, probs = self._buf("logits", (D, H, W), F32), self._buf("probs", (D, H, W), F32)
        if W % 8 == 0 and self.rows8:
            ops.conv3d_rows8_final(a1, self._pk("out2/f/rows8", "output_layer.2.weight", rows8_weight_image),
                                   p["output_layer.2.bias"], logits, probs)
        elif W % 16 == 0:
            ops.conv3d_wpack8_final(a1, self._pk("out2/f/wpack", "output_layer.2.weight", lambda w_: wpack_weight_image(w_, 16)),
                                    p["output_layer.2.bias"].repeat(16).contiguous(), logits, probs)
        else:
            ops.head_out_conv(a1, p["output_layer.2.weight"].permute(2, 3, 4, 0, 1).reshape(27, 8).contiguous(),
                              p["output_layer.2.bias"], logits, probs)
        lab = self._buf("labels", (D, H, W), F32)
        lab.copy_(labels.to(dev))
        stats8 = ops.seg_stats(probs, lab)
        loss = 1.0 - 2.0 * stats8[2] / (stats8[1] + stats8[0] + 1e-3)
        self.launches += 4
        # ---------------- backward
        dl8 = self._buf("dlogit8", (D, H, W, 8))
        T.dice_bwd(logits, probs, lab, stats8, dl8, grad_scale)
        # output_layer.2 (8 -> 1): operate on the 8-channel padded gradient (channel 0 live)
        dw2 = T.conv_weight_gradient(a1, dl8, 1, self._bufs.setdefault("wgrad_pool", {}))  # [27, 8 (co, only 0 live), 8 (ci)]
        g["output_layer.2.weight"].copy_(dw2[:, 0].view(3, 3, 3, 8).permute(3, 0, 1, 2)[None])
        db2 = torch.zeros(8, device=dev, dtype=F32)
        T.colsum(dl8, db2)
        g["output_layer.2.bias"].copy_(db2[:1])
        # forward weight zero-padded to 8 output channels (the gradient volume carries 8 channels, channel 0 live)
        c_out2 = _Conv(self, "output_layer.2.weight", 8, 8, 1,
                       pre=lambda w_: torch.cat([w_, torch.zeros(7, 8, 3, 3, 3, device=w_.device, dtype=w_.dtype)]))
        dz1 = self._buf("dz_o0", (D, H, W, 8))
        if fuse_bwd:
            c_out2.input_gradient(dl8, dz1, z_below=z1)
            self._bias_grad(dz1, "output_layer.0.bias")
        else:
            self._dgrad_gelu(c_out2, dl8, z1, dz1, "output_layer.0.bias", "da_o0")
        self._wgrad_conv(cur, dz1, 1, "output_layer.0.weight")
        dcur = self._buf("d_top", (D, H, W, 8))  # d(at) of the last block, or (fused) already d(zt)
        co.input_gradient(dz1, dcur, z_below=saved[3][10] if fuse_bwd else None)
        dcur_is_dz = fuse_bwd
        dzun_ready = False
        self.launches += 14
        for bi in reversed(range(4)):
            c1, c2, c3, d1, d2 = BLOCKS[bi]
            pre = f"layers.{bi + 2}.layers."
            blk_in, n_out, stats, G, ca, za, aa, cb, zb, ab, zt, at, H, W = saved[bi]
            # transposed convolution: dcur is d(at) [D, 2H, 2W, c3]
            dzun = self._buf(f"dzun{bi}", (D, H, W, 4 * c3))
            if dzun_ready:  # the GroupNorm backward of the block above already wrote d(zt), unshuffled, and the bias gradient
                dzun_ready = False
            elif dcur_is_dz:  # the producer's epilogue already applied gelu'(zt)
                self._bias_grad(dcur, pre + "5.bias")
                T.pixel_unshuffle(dcur, dzun)
                dcur_is_dz = False
            else:
                # d(zt) = d(at) * gelu'(zt), written straight in the sub-pixel-major row layout of the GEMMs below; the bias
                # gradient (summed over voxels AND sub-pixels) from the same pass
                db = torch.zeros(c3, device=dev, dtype=F32)
                T.gelu_bwd_unshuffle(dcur, zt, dzun, db)
                g[pre + "5.bias"].copy_(db)
            rows = D * H * W
            dwt = self._wgrad_rows(ab.view(rows, c2), dzun.view(rows, 4 * c3))          # [(ij, c3), c2]
            g[pre + "5.weight"].copy_(dwt.view(2, 2, c3, c2).permute(3, 2, 0, 1)[:, :, None])
            n_pad = max(32, c2)  # dX = dZun @ wd^T, wd = the weight as [c2, (i, j, co)], zero rows up to the MMA N tile

            def wd_fn(wT, c2_=c2, c3_=c3, n_=n_pad):
                wd = wT[:, :, 0].permute(0, 2, 3, 1).reshape(c2_, 4 * c3_)
                return torch.cat([wd, torch.zeros(n_ - c2_, 4 * c3_, device=wT.device, dtype=wT.dtype)]) if n_ > c2_ else wd

            wd_p = self._pk(pre + "5/g", pre + "5.weight", wd_fn)
            dzb = self._buf(f"dzb{bi}", (D, H, W, c2))
            dza = self._buf(f"dza{bi}", (D, H, W, c2))
            zero_b = torch.zeros(n_pad, device=dev, dtype=F32)
            if fuse_bwd:
                # conv b, conv a: each input gradient leaves its epilogue as the gradient of the pre-activation below
                T.linear_nvalid(dzun.view(rows, 4 * c3), wd_p, zero_b, dzb.view(rows, c2), c2, z=zb.view(rows, c2))
                self._bias_grad(dzb, pre + "3.bias")
                self._wgrad_conv(aa, dzb, d2, pre + "3.weight")
                cb.input_gradient(dzb, dza, z_below=za)
                self._bias_grad(dza, pre + "1.bias")
            else:
                dab = self._buf(f"dab{bi}", (D, H, W, c2))
                T.linear_nvalid(dzun.view(rows, 4 * c3), wd_p, zero_b, dab.view(rows, c2), c2)
                # conv b
                self._gelu_bwd_bias(dab, zb, dzb, pre + "3.bias")
                self._wgrad_conv(aa, dzb, d2, pre + "3.weight")
                # conv a
                self._dgrad_gelu(cb, dzb, za, dza, pre + "1.bias", f"daa{bi}")
            self._wgrad_conv(n_out, dza, d1, pre + "1.weight")
            dn = self._buf(f"dn{bi}", (D, H, W, c1))
            ca.input_gradient(dza, dn)
            # GroupNorm
            dgam, dbet = torch.empty(c1, device=dev, dtype=F32), torch.empty(c1, device=dev, dtype=F32)
            if self.fuse_gn_gelu:
                # the block's input is gelu(z) of the layer below (a transposed convolution, or the projection): its GELU
                # backward, bias gradient and (transposed convolution) pixel-unshuffle ride on the GroupNorm backward's pass
                db = torch.zeros(c1, device=dev, dtype=F32)
                if bi > 0:
                    c3p = BLOCKS[bi - 1][2]
                    dz_below = self._buf(f"dzun{bi - 1}", (D, H // 2, W // 2, 4 * c3p))
                    T.groupnorm_bwd_gelu(blk_in, dn, dz_below, p[pre + "0.weight"], stats, dgam, dbet, G, 1e-3, saved[bi - 1][10], db, True)
                    g[f"layers.{bi + 1}.layers.5.bias"].copy_(db)
                    dzun_ready = True
                else:
                    dzp = self._buf("dz_proj", (vox, 1024))
                    T.groupnorm_bwd_gelu(blk_in, dn, dzp.view(D, H, W, 1024), p[pre + "0.weight"], stats, dgam, dbet, G, 1e-3,
                                         z_proj.view(D, H, W, 1024), db, False)
                    g["layers.0.bias"].copy_(db)
            else:
                dblk = self._buf(f"dblk{bi}", (D, H, W, c1))
                T.groupnorm_bwd(blk_in, dn, dblk, p[pre + "0.weight"], stats, dgam, dbet, G, 1e-3)
                dcur = dblk
            g[pre + "0.weight"].copy_(dgam)
            g[pre + "0.bias"].copy_(dbet)
            self.launches += 14
        # projection (1x1x1): only the weight / bias gradient (the features are data)
        dzp = self._buf("dz_proj", (vox, 1024))
        if not self.fuse_gn_gelu:
            self._gelu_bwd_bias(dcur.view(vox, 1024), z_proj, dzp, "layers.0.bias")
        if cfirst:
            dw0 = self._wgrad_rows(None, dzp, xt=feats.view(C, vox).to(BF16))
        else:
            dw0 = self._wgrad_rows(x0.view(vox, C), dzp)
        g["layers.0.weight"].copy_(dw0.view(1024, C, 1, 1, 1))
        self.launches += 2
        return loss

    def optimizer_step(self) -> None:
        """Data-parallel: sum the flat gradient bucket over the ranks (one NCCL all-reduce; the 1/world factor was
        applied to the loss gradient), then AdamW on the fp32 master weights."""
        allreduce_gradient_bucket(self.flat_g)
        self.step_count += 1
        T.adamw(self.flat_p, self.flat_g, self.flat_m, self.flat_v, self.lr, self.betas[0], self.betas[1], self.eps,
                self.weight_decay, self.step_count)
        self.launches += 1

    def train_step(self, features: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        import torch.distributed as dist

        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        with nvtx.span("head.train.forward_backward"):
            loss = self._forward_backward_graphed(features, labels, 1.0 / world)
        with nvtx.span("head.train.optimizer"):
            self.optimizer_step()
        return loss

    # ----------------------------------------------------------------------------- CUDA graph of forward + backward
    def _forward_backward_graphed(self, features: torch.Tensor, labels: torch.Tensor, grad_scale: float) -> torch.Tensor:
        """forward_backward is ~200 kernels of ours plus the small torch kernels that re-pack the updated weights:
        launch-bound for a fifth of the step. The first two steps of a given crop shape run eagerly (first-use
        allocations, attribute settings, lookup tables); the third is captured into a CUDA graph over static input
        buffers and every later step replays it. The all-reduce and AdamW (whose bias correction takes the step number
        by value) stay outside the graph. CVIT_TRAIN_GRAPH=0 or a failed capture falls back to eager launches."""
        import os

        if os.environ.get("CVIT_TRAIN_GRAPH", "1") == "0" or self._graph_broken:
            return self.forward_backward(features, labels, grad_scale)
        key = (tuple(features.shape), features.dtype, tuple(labels.shape), labels.dtype, float(grad_scale))
        ent = self._graphs.get(key)
        if ent is None:
            if len(self._graphs) >= 2:  # every graph keeps its own pool of temporaries: only the two commonest crop shapes
                return self.forward_backward(features, labels, grad_scale)
            ent = self._graphs[key] = {"seen": 0}
        if "graph" not in ent:
            ent["seen"] += 1
            if ent["seen"] <= 2:
                return self.forward_backward(features, labels, grad_scale)
            try:
                ent["f"] = torch.empty(features.shape, device=self.device, dtype=features.dtype)
                ent["l"] = torch.empty(labels.shape, device=self.device, dtype=labels.dtype)
                ent["f"].copy_(features, non_blocking=True)
                ent["l"].copy_(labels, non_blocking=True)
                torch.cuda.synchronize()
                l0 = self.launches
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    ent["loss"] = self.forward_backward(ent["f"], ent["l"], grad_scale)
                ent["launches"] = self.launches - l0
                self.launches = l0
                ent["graph"] = graph
            except Exception as e:  # noqa: BLE001  (capture is an optimisation: never fatal)
                import logging

                logging.warning("CUDA-graph capture of the training step failed (%s: %s); running eagerly", type(e).__name__, e)
                self._graph_broken = True
                torch.cuda.synchronize()
                return self.forward_backward(features, labels, grad_scale)
        ent["f"].copy_(features, non_blocking=True)
        ent["l"].copy_(labels, non_blocking=True)
        ent["graph"].replay()
        self.launches += ent["launches"]
        return ent["loss"]
