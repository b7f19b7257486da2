"""B200-native CryoVIT 3-D segmentation head (reference src/cryovit/models/cryovit.py:10-83).

``CryoVITHeadB200`` keeps the reference's parameter names (``layers.0.weight``, ``layers.2.layers.1.weight``, ...,
``output_layer.2.bias``), so a reference ``weights.pt`` loads unchanged (eval_model.py:185-186), and mirrors its
call surface: ``forward_volume(x[B,C,D,h,w]) -> clipped logits [B,1,D,16h,16w]`` and
``forward(batch) -> probabilities [B,D,16h,16w]``.

Device layout: every intermediate volume is channels-last bf16 ``[D, H, W, C]``; convolutions are implicit GEMMs on
tcgen05 (TMA box loads whose out-of-bounds zero fill is the "same" padding), ConvTranspose(1,2,2) is a GEMM with a
pixel-shuffle store. GroupNorm never touches the volume on its own: its statistics come out of the epilogue of the
layer that produces its input, its scale is folded into the weights of the convolution that follows and its shift into
a 64-row border-aware bias table (csrc/gn_fold.cu); ``fuse_groupnorm=False`` keeps the two-pass kernel (A/B, tests).
``in_channels`` generalises the reference's hard-wired 1536 (BASELINE config 1 feeds ViT-S features, 384).
"""
from __future__ import annotations

import torch

from . import ops
from ._lib import CryovitB200Error
from .operand_gather import OperandGather

BLOCKS = [(1024, 192, 128, 32, 24), (128, 64, 32, 16, 12), (32, 32, 32, 8, 4), (32, 16, 8, 2, 1)]


def state_dict_keys() -> list[str]:
    keys = ["layers.0.weight", "layers.0.bias"]
    for bi in range(4):
        for li in (0, 1, 3, 5):
            keys += [f"layers.{bi + 2}.layers.{li}.weight", f"layers.{bi + 2}.layers.{li}.bias"]
    return keys + ["output_layer.0.weight", "output_layer.0.bias", "output_layer.2.weight", "output_layer.2.bias"]


def _conv_taps(w: torch.Tensor, cout_pad: int) -> torch.Tensor:
    """Conv3d weight [Cout, Cin, 3, 3, 3] -> [27 * cout_pad, Cin], tap = (kd*3 + kh)*3 + kw."""
    cout, cin = w.shape[:2]
    wt = torch.zeros(27, cout_pad, cin, dtype=w.dtype)
    wt[:, :cout] = w.permute(2, 3, 4, 0, 1).reshape(27, cout, cin)
    return wt.reshape(27 * cout_pad, cin)


def halo_weight_image(w: torch.Tensor, cout_pad: int) -> torch.Tensor:
    """Conv3d weight [Cout, Cin, 3, 3, 3] (Cin in {8, 16, 32}) -> the shared-memory image csrc/conv_halo.cu keeps
    resident: [kd*3+kh][mma][2 K chunks][cout_pad][8 channels]. For Cin >= 16 MMA i is (tap kw = i // (Cin/16),
    16-channel step c2 = i % (Cin/16)) and its K chunks are the two halves of those 16 channels; for Cin == 8 an MMA
    covers two neighbouring taps: (kw0, kw1), then (kw1 with zero weights, kw2)."""
    cout, cin = w.shape[:2]
    steps = cin // 16
    n_mma = 3 * steps if cin >= 16 else 2
    img = torch.zeros(9, n_mma, 2, cout_pad, 8, dtype=torch.float32)
    wt = w.float().permute(2, 3, 4, 0, 1).reshape(9, 3, cout, cin)  # [kd*3+kh][kw][co][ci]
    if cin >= 16:
        for i in range(n_mma):
            kw, c2 = divmod(i, steps)
            for k in range(2):
                img[:, i, k, :cout] = wt[:, kw, :, c2 * 16 + k * 8: c2 * 16 + k * 8 + 8]
    else:
        img[:, 0, 0, :cout] = wt[:, 0]
        img[:, 0, 1, :cout] = wt[:, 1]
        img[:, 1, 1, :cout] = wt[:, 2]  # chunk 0 of the second MMA re-reads tap kw1 against zero weights
    return img.reshape(-1)


def wpackn_weight_image(w: torch.Tensor, cout_pad: int, P: int) -> torch.Tensor:
    """Conv3d weight [Cout, Cin, 3, 3, 3] (Cin 16 or 32) -> the banded shared-memory image of csrc/conv_wpackn.cu (fp32, flat):
    [kd*3+kh][K step][2 chunks][n = j_out * cout_pad + co][8], where chunk k = 2 step + c is (window voxel j_in, channel
    chunk c_hi) = divmod(k, Cin / 8) -- the window of a group of P output voxels starts one voxel to their left -- and the
    entry is w[co, c_hi*8 + e, kd, kh, kw] with kw = j_in - j_out when that is a tap (0..2), zero otherwise."""
    cout, cin = w.shape[:2]
    ch = cin // 8
    wt = torch.zeros(9, 3, cout_pad, ch, 8, device=w.device)
    wt[:, :, :cout] = w.float().permute(2, 3, 4, 0, 1).reshape(9, 3, cout, ch, 8)
    img = torch.zeros(9, P + 2, ch, P, cout_pad, 8, device=w.device)
    for j_out in range(P):
        for kw in range(3):
            img[:, j_out + kw, :, j_out] = wt[:, kw].permute(0, 2, 1, 3)  # [9, ch, cout_pad, 8]
    return img.reshape(-1)


_BANDS: dict = {}


def wpack_weight_image(w: torch.Tensor, P: int) -> torch.Tensor:
    """Conv3d weight [Cout, 8, 3, 3, 3] -> the banded shared-memory image of csrc/conv_wpack.cu:
    [kh][K step][2 chunks][block: kd = 2, 1, 0][n = j_out * Cout + co][8 ci], where chunk c of step s is window voxel
    j_in = 2 s + c (the window of a group of P output voxels starts one voxel to their left) and the entry is
    w[co, ci, kd, kh, kw] with kw = j_in - j_out when that is a tap (0..2), zero otherwise. The three depth taps are
    stacked along the MMA N dimension in the order of the output depths they feed (p-1, p, p+1 for input plane p)."""
    cout, cin = w.shape[:2]
    assert cin == 8 and (P + 2) % 2 == 0
    wt = w.float().permute(2, 3, 4, 0, 1)  # [kd][kh][kw][co][ci], on w's device
    key = (P, str(w.device))
    band = _BANDS.get(key)
    if band is None:  # band[j_in, j_out, kw] = 1 where kw == j_in - j_out (built once per device: no host copies later)
        band = torch.zeros(P + 2, P, 3)
        for kw in range(3):
            band[torch.arange(P) + kw, torch.arange(P), kw] = 1.0
        band = _BANDS[key] = band.to(w.device)
    # [kh][j_in][kd][j_out][co][ci] -> blocks in the order kd = 2, 1, 0 -> j_in split into (K step, chunk)
    img = torch.einsum("jok,dhkcx->hjdocx", band, wt).flip(2)
    return img.reshape(3, (P + 2) // 2, 2, 3, P, cout, 8).reshape(-1)


def rows8_weight_image(w: torch.Tensor) -> torch.Tensor:
    """Conv3d weight [8, 8, 3, 3, 3] -> the shared-memory image of csrc/conv_rows8.cu (fp32, flat):
    [v = input plane mod 3][K step][chunk][96 rows][8 ci]. Row n = (yr * 3 + p) * 8 + co holds
    w[co, ci, kd, kh = 2 - yr, kw] with kw = 2 * step + chunk (the fourth tap is zero) and kd = (v + 1 - p) mod 3: an input
    row (z', y') feeds output row y' - 1 + yr of the output plane whose slot is p = (z' - (kd - 1)) mod 3. Rows 72..95 are zero."""
    cout, cin = w.shape[:2]
    assert cout <= 8 and cin == 8
    img = torch.zeros(3, 2, 2, 96, 8, device=w.device)
    wf = w.float()
    for v in range(3):
        for yr in range(3):
            for p_ in range(3):
                kd, kh = (v + 1 - p_) % 3, 2 - yr
                n0 = (yr * 3 + p_) * 8
                for kw in range(3):
                    img[v, kw // 2, kw % 2, n0:n0 + cout] = wf[:, :, kd, kh, kw]
    return img.reshape(-1)


def rowsn_weight_image(w: torch.Tensor) -> torch.Tensor:
    """Conv3d weight [Cout, Cin, 3, 3, 3] (Cin, Cout in {16, 32}) -> the shared-memory images of csrc/conv_rows.cu (fp32, flat):
    [pass h = co // 16][rotation v][chunk j = ci // 8][K step][chunk c][144 rows][8]; row = (yr * 3 + slot) * 16 + co % 16 holds
    w[co, j*8 + e, kd, kh = 2 - yr, kw = 2 step + c] with kd = (v + 1 - slot) mod 3 (the fourth column tap is zero)."""
    cout, cin = w.shape[:2]
    assert cin in (16, 32) and cout in (16, 32)
    wf = w.float().reshape(cout // 16, 16, cin // 8, 8, 3, 3, 3)  # [h][col][j][e][kd][kh][kw]
    img = torch.zeros(cout // 16, 3, cin // 8, 2, 2, 144, 8, device=w.device)
    for v in range(3):
        for yr in range(3):
            for slot in range(3):
                kd, kh = (v + 1 - slot) % 3, 2 - yr
                n0 = (yr * 3 + slot) * 16
                for kw in range(3):
                    img[:, v, :, kw // 2, kw % 2, n0:n0 + 16] = wf[:, :, :, :, kd, kh, kw].permute(0, 2, 1, 3)
    return img.reshape(-1)


class CryoVITHeadB200:
    def __init__(self, in_channels: int = 1536, fuse_groupnorm: bool | None = None, wpack_narrow: bool | None = None):
        import os

        self.in_channels = in_channels
        # None: on, unless the environment says otherwise (A/B runs: CVIT_HEAD_FUSE_GN=0, CVIT_HEAD_WPACKN=0)
        self.fuse_groupnorm = os.environ.get("CVIT_HEAD_FUSE_GN", "1") != "0" if fuse_groupnorm is None else fuse_groupnorm
        # False: the 16- / 32-channel layers run on the per-tap halo kernel
        self.wpack_narrow = os.environ.get("CVIT_HEAD_WPACKN", "1") != "0" if wpack_narrow is None else wpack_narrow
        self.rows8 = os.environ.get("CVIT_HEAD_ROWS8", "1") != "0"  # the two 8-channel output convolutions on conv_rows8.cu
        self.rowsn = os.environ.get("CVIT_HEAD_ROWSN", "1") != "0"  # the 16 / 32-channel layers on conv_rows.cu (else W-packed)
        self.device: torch.device | None = None
        self._sd_cpu: dict | None = None
        self._w: dict = {}
        self._bufs: dict = {}
        self._bucket = None  # attach_bucket: (OperandGather, index-valued operand tree, id -> operand name, projection range)
        self.launches = 0

    # ----------------------------------------------------------------------------- nn.Module-like surface
    def load_state_dict(self, sd: dict, strict: bool = True):
        missing = [k for k in state_dict_keys() if k not in sd]
        if strict and missing:
            raise CryovitB200Error(f"head state dict is missing {missing[:3]} ...")
        if sd["layers.0.weight"].shape[1] != self.in_channels:
            raise CryovitB200Error(f"layers.0.weight expects {sd['layers.0.weight'].shape[1]} input channels, "
                                   f"head was built for {self.in_channels}")
        self._sd_cpu = {k: v.detach().float().cpu() for k, v in sd.items()}
        if self.device is not None:
            self._pack()
        return self

    def state_dict(self) -> dict:
        return dict(self._sd_cpu or {})

    def cuda(self, device=None):
        if not torch.cuda.is_available():
            raise CryovitB200Error("no CUDA device: the B200 hot path has no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        if self._sd_cpu is not None:
            self._pack()
        return self

    def eval(self):
        return self

    def _pack(self, sd: dict | None = None, gather: OperandGather | None = None) -> tuple[dict, dict]:
        """Every operand of the forward pass from the (CPU, fp32) state dict ``sd`` (default: the loaded one). With
        ``gather``, ``sd`` holds index-valued stand-ins of the parameters (``OperandGather.indices``): each operand is
        registered there as a gather table, and the returned tree holds the index-valued operands (``attach_bucket``).
        Returns (operand tree, id of each gathered operand -> its name in ``gather``)."""
        dev = self.device
        ids = {}

        def cast(t, dtype):
            if gather is None:
                return t.to(dev).to(dtype).contiguous()
            t = t.to(dev).float().contiguous().clone()
            ids[id(t)] = name = str(len(ids))
            gather.add(name, t, dtype)
            return t

        if sd is None:
            sd = self._sd_cpu
        bf = lambda t: cast(t, torch.bfloat16)
        f32 = lambda t: cast(t, torch.float32)
        w = {"proj_w": bf(sd["layers.0.weight"].reshape(1024, self.in_channels)), "proj_b": f32(sd["layers.0.bias"])}
        pw = sd["layers.0.weight"].reshape(1024, self.in_channels).float()
        if gather is not None or float(pw.abs().max()) < 6.0e4:  # fp16 image of the projection for the transposed-A kernel
            w["proj_w16"] = cast(pw, torch.float16)                # (fp16 features); with gather, checked per refresh
        blocks = []
        for bi, (c1, c2, c3, d1, d2) in enumerate(BLOCKS):
            p = f"layers.{bi + 2}.layers."
            c2p = max(32, c2)  # MMA N tile is a multiple of 32: zero-pad 16 -> 32 output channels
            ba, bb = torch.zeros(c2p), torch.zeros(c2p)
            ba[:c2], bb[:c2] = sd[p + "1.bias"], sd[p + "3.bias"]
            wT = sd[p + "5.weight"]  # [c2, c3, 1, 2, 2]
            halo, wpn, rws = {}, {}, {}
            for tag, key, cin in (("a", "1", c1), ("b", "3", c2)):
                if ops.rows_supported(cin, c2):  # one voxel per tensor-core row (csrc/conv_rows.cu): the 16 / 32-channel layers
                    img32 = f32(rowsn_weight_image(sd[p + key + ".weight"]))
                    rws[tag] = {"w32": img32, "w": bf(img32), "bias": f32(sd[p + key + ".bias"]),
                                "table": f32(sd[p + key + ".bias"].repeat(64)), "fold": torch.empty_like(img32, dtype=torch.bfloat16),
                                "gn_table": torch.empty(64 * c2, device=dev, dtype=torch.float32)}
                if cin in (8, 16, 32):  # narrow layer: shared-memory halo kernel (csrc/conv_halo.cu)
                    cp = 32 if c2 > 16 else 16
                    hb = torch.zeros(cp)
                    hb[:c2] = sd[p + key + ".bias"]
                    halo[tag] = (bf(halo_weight_image(sd[p + key + ".weight"], cp)), f32(hb), cp)
                    P = ops.wpackn_group(cin, cp)
                    if P:  # ... or, on planes whose width is a multiple of P, P voxels per tensor-core row (csrc/conv_wpackn.cu)
                        img32 = f32(wpackn_weight_image(sd[p + key + ".weight"], cp, P))
                        wpn[tag] = {"P": P, "cp": cp, "w32": img32, "w": bf(img32),
                                    "table": f32(hb.repeat(64)), "fold": torch.empty_like(img32, dtype=torch.bfloat16)}
            # fp32 originals in the operand layout of the convolution that follows the GroupNorm (folded per volume)
            if "a" in halo:
                a32, a_layout, a_cp = f32(halo_weight_image(sd[p + "1.weight"], halo["a"][2])), ops.LAYOUT_HALO, halo["a"][2]
                a_bias = halo["a"][1]
            else:
                a32, a_layout, a_cp, a_bias = f32(_conv_taps(sd[p + "1.weight"], c2p).reshape(-1)), ops.LAYOUT_TAPS, c2p, f32(ba)
            blocks.append({
                "wpn": wpn, "rows": rws,
                "halo": halo, "a_w32": a32, "a_layout": a_layout, "a_cp": a_cp, "a_bias": a_bias,
                "a_fold": torch.empty(a32.numel(), device=dev, dtype=torch.bfloat16),
                "a_table": torch.empty(64 * a_cp, device=dev, dtype=torch.float32),
                "gn_ab": ops.groupnorm_fold_ab(c1, max(8, c1 // 8), dev),
                "groups": max(8, c1 // 8), "gn_w": f32(sd[p + "0.weight"]), "gn_b": f32(sd[p + "0.bias"]),
                "a_w": bf(_conv_taps(sd[p + "1.weight"], c2p)), "a_b": f32(ba), "d1": d1,
                "b_w": bf(_conv_taps(sd[p + "3.weight"], c2p)), "b_b": f32(bb), "d2": d2,
                "t_w": bf(wT[:, :, 0].permute(2, 3, 1, 0).reshape(4 * c3, c2)), "t_b": f32(sd[p + "5.bias"].repeat(4)),
                "c1": c1, "c2": c2, "c3": c3,
            })
        w["blocks"] = blocks
        o1b = torch.zeros(16)
        o1b[:8] = sd["output_layer.0.bias"]
        w["o1_img"], w["o1_b16"] = bf(halo_weight_image(sd["output_layer.0.weight"], 16)), f32(o1b)
        w["o2_w"] = f32(sd["output_layer.2.weight"].permute(2, 3, 4, 0, 1).reshape(27, 8))
        w["o2_b"] = f32(sd["output_layer.2.bias"])
        # W-packed tensor-core versions of both output convolutions (planes whose width is a multiple of 16)
        w["o1_wp"], w["o1_wp_b"] = bf(wpack_weight_image(sd["output_layer.0.weight"], 8)), f32(sd["output_layer.0.bias"].repeat(8))
        w["o2_wp"], w["o2_wp_b"] = bf(wpack_weight_image(sd["output_layer.2.weight"], 16)), f32(sd["output_layer.2.bias"].repeat(16))
        # one voxel per MMA row, partial sums meeting in tensor memory (csrc/conv_rows8.cu; widths that are a multiple of 8)
        w["o1_r8"], w["o1_r8_b"] = bf(rows8_weight_image(sd["output_layer.0.weight"])), f32(sd["output_layer.0.bias"])
        w["o2_r8"], w["o2_r8_b"] = bf(rows8_weight_image(sd["output_layer.2.weight"])), f32(sd["output_layer.2.bias"])
        if gather is None:
            self._w = w
        return w, ids

    # ----------------------------------------------------------------------------- weights that follow a trainer
    def attach_bucket(self, store: torch.Tensor, offsets: dict[str, int], shapes: dict[str, tuple]) -> "CryoVITHeadB200":
        """Take the weights from a flat fp32 parameter bucket (``CryoVITHeadTrainerB200.parameter_bucket()``: the
        parameters at ``offsets`` with ``shapes``, a zero at the end) instead of a state dict. ``_pack`` runs ONCE, on
        the parameters' global indices, and leaves a gather table per operand; every :meth:`refresh` then rebuilds all
        operands from the bucket's current values with one ``index_select`` per dtype, no host round trip."""
        if self.device is None:
            raise CryovitB200Error("attach_bucket: call .cuda() first")
        if shapes["layers.0.weight"][1] != self.in_channels:
            raise CryovitB200Error(f"bucket's layers.0.weight expects {shapes['layers.0.weight'][1]} input channels, "
                                   f"head was built for {self.in_channels}")
        gather = OperandGather(store)
        sd = {k: gather.indices(offsets[k], shapes[k], device="cpu") for k in state_dict_keys()}
        tree, ids = self._pack(sd, gather)
        o = offsets["layers.0.weight"]
        self._bucket = (gather, tree, ids, (o, o + 1024 * self.in_channels))
        self._sd_cpu = None  # the weights now live in the bucket
        return self.refresh()

    def refresh(self) -> "CryoVITHeadB200":
        """Operands from the attached bucket's current values. The fp16 projection (fp16 features) exists while the
        projection weight fits in fp16, as with ``load_state_dict``: one host read per refresh."""
        if self._bucket is None:
            raise CryovitB200Error("refresh: no bucket attached (attach_bucket)")
        gather, tree, ids, (p0, p1) = self._bucket
        views = gather.refresh()

        def sub(x):
            if isinstance(x, dict):
                return {k: sub(v) for k, v in x.items()}
            if isinstance(x, (list, tuple)):
                return type(x)(sub(v) for v in x)
            if isinstance(x, torch.Tensor) and id(x) in ids:
                return views[ids[id(x)]]
            return x

        w = sub(tree)
        if not float(gather.store[p0:p1].abs().max()) < 6.0e4:
            del w["proj_w16"]
        self._w = w
        return self

    def _buf(self, name: str, numel: int, dtype=torch.bfloat16) -> torch.Tensor:
        b = self._bufs.get(name)
        if b is None or b.numel() < numel or b.dtype != dtype:
            b = torch.empty(numel, device=self.device, dtype=dtype)
            self._bufs[name] = b
        return b[:numel]

    # ----------------------------------------------------------------------------- forward
    def _trunk(self, features: torch.Tensor):
        """Every layer before output_layer: features (C, D, h, w) -> (bf16 [D, 16h, 16w, 8] in one of the ping-pong
        buffers, the name of the other one)."""
        if self.device is None or not self._w:
            raise CryovitB200Error("head not ready: call load_state_dict(...) and .cuda() first")
        if features.dim() != 4 or features.shape[0] != self.in_channels:
            raise CryovitB200Error(f"expected features (C={self.in_channels}, D, h, w), got {tuple(features.shape)}")
        C, D, h, w = features.shape
        w_ = self._w
        y = self._buf("pong", D * h * w * 1024).view(D * h * w, 1024)
        vox0 = D * h * w
        fuse = self.fuse_groupnorm
        blocks = w_["blocks"]
        # GroupNorm statistics ride on the producer of each normalised tensor: [32-row block][group (x sub-pixel)][2]
        cpg = [b["c1"] // b["groups"] for b in blocks]
        partials = None
        if fuse:
            need = ops.gn_partials_numel(vox0, 1024, cpg[0])
            Hc, Wc = h, w
            for bi in range(len(blocks) - 1):
                need = max(need, ops.gn_partials_numel(D * Hc * Wc, 4 * blocks[bi]["c3"], cpg[bi + 1]), 16 * 256 * 1024)
                Hc, Wc = 2 * Hc, 2 * Wc
            partials = self._buf("gn_partials", need, torch.float32)
        if features.dtype == torch.float16 and "proj_w16" in w_ and vox0 % 8 == 0 and C % 8 == 0 and C >= 64:
            # the on-disk layout (C, D*h*w) IS the A operand (MN-major): no channels-last copy of the features
            if fuse:
                ops.linear_bias_cfirst_gn(features.contiguous().view(C, vox0), w_["proj_w16"], w_["proj_b"], y, partials, cpg[0])
            else:
                ops.linear_bias_cfirst(features.contiguous().view(C, vox0), w_["proj_w16"], w_["proj_b"], y, gelu=True)
            self.launches += 1
        else:
            x = self._buf("ping", vox0 * max(C, 1024)).narrow(0, 0, vox0 * C).view(D, h, w, C)
            ops.features_to_ndhwc(features.contiguous(), x)
            if fuse:
                ops.linear_bias_gelu_gn(x.view(vox0, C), w_["proj_w"], w_["proj_b"], y, partials, cpg[0])
            else:
                ops.linear_bias(x.view(vox0, C), w_["proj_w"], w_["proj_b"], y, gelu=True)
            self.launches += 2
        cur, H, W = y.view(D, h, w, 1024), h, w
        stats = self._buf("gn_stats", 256, torch.float32)
        names = ["ping", "pong"]
        flip = 0  # cur lives in "pong"
        prod_rows, prod_cols = vox0, 1024  # GEMM rows / columns of the layer that produced `cur`
        for bi, b in enumerate(blocks):
            c1, c2, c3 = b["c1"], b["c2"], b["c3"]
            vox = D * H * W
            nxt = self._buf(names[flip], vox * c2).view(D, H, W, c2)
            ra = b["rows"].get("a") if self.rowsn else None
            rb = b["rows"].get("b") if self.rowsn else None
            wa = b["wpn"].get("a") if ra is None and self.wpack_narrow and "a" in b["wpn"] and W % b["wpn"]["a"]["P"] == 0 else None
            wb = b["wpn"].get("b") if rb is None and self.wpack_narrow and "b" in b["wpn"] and W % b["wpn"]["b"]["P"] == 0 else None
            if fuse:
                # statistics -> scale / shift -> folded weights + border-aware bias table -> convolution of the RAW tensor
                if ra is not None:
                    ops.groupnorm_fold(partials, prod_rows, prod_cols // cpg[bi], b["groups"], vox * cpg[bi], b["gn_w"], b["gn_b"], 1e-3,
                                       b["gn_ab"], ra["w32"], ra["fold"], c1, c2, ops.LAYOUT_ROWS, ra["bias"], ra["gn_table"])
                    ops.conv3d_rows(cur, ra["fold"], ra["gn_table"], nxt, b["d1"])
                elif wa is not None:
                    ops.groupnorm_fold(partials, prod_rows, prod_cols // cpg[bi], b["groups"], vox * cpg[bi], b["gn_w"], b["gn_b"], 1e-3,
                                       b["gn_ab"], wa["w32"], wa["fold"], c1, wa["cp"], ops.LAYOUT_WPACKN, b["a_bias"], b["a_table"])
                    ops.conv3d_wpackn(cur, wa["fold"], b["a_table"], nxt, b["d1"], wa["cp"])
                else:
                    ops.groupnorm_fold(partials, prod_rows, prod_cols // cpg[bi], b["groups"], vox * cpg[bi], b["gn_w"], b["gn_b"], 1e-3,
                                       b["gn_ab"], b["a_w32"], b["a_fold"], c1, b["a_cp"], b["a_layout"], b["a_bias"], b["a_table"])
                if wa is not None or ra is not None:
                    pass
                elif "a" in b["halo"]:
                    ops.conv3d_halo_tab(cur, b["a_fold"], b["a_table"], nxt, b["d1"], b["a_cp"])
                else:
                    ops.conv3d_dilated_tab(cur, b["a_fold"].view(27 * b["a_cp"], c1), b["a_table"], nxt, b["d1"])
            else:
                ops.groupnorm_ndhwc(cur, cur, b["gn_w"], b["gn_b"], stats[: 2 * b["groups"]], b["groups"], 1e-3)
                if ra is not None:
                    ops.conv3d_rows(cur, ra["w"], ra["table"], nxt, b["d1"])
                elif wa is not None:
                    ops.conv3d_wpackn(cur, wa["w"], wa["table"], nxt, b["d1"], wa["cp"])
                elif "a" in b["halo"]:
                    ops.conv3d_halo(cur, b["halo"]["a"][0], b["halo"]["a"][1], nxt, b["d1"], b["halo"]["a"][2])
                else:
                    ops.conv3d_dilated(cur, b["a_w"], b["a_b"], nxt, b["d1"])
            cur, flip = nxt, flip ^ 1
            nxt = self._buf(names[flip], vox * c2).view(D, H, W, c2)
            if rb is not None:
                ops.conv3d_rows(cur, rb["w"], rb["table"], nxt, b["d2"])
            elif wb is not None:
                ops.conv3d_wpackn(cur, wb["w"], wb["table"], nxt, b["d2"], wb["cp"])
            elif "b" in b["halo"]:
                ops.conv3d_halo(cur, b["halo"]["b"][0], b["halo"]["b"][1], nxt, b["d2"], b["halo"]["b"][2])
            else:
                ops.conv3d_dilated(cur, b["b_w"], b["b_b"], nxt, b["d2"])
            cur, flip = nxt, flip ^ 1
            nxt = self._buf(names[flip], 4 * vox * c3).view(D, 2 * H, 2 * W, c3)
            if fuse and bi + 1 < len(blocks):
                prod_rows, prod_cols = ops.convT_1x2x2_gn(cur, b["t_w"], b["t_b"], nxt, partials, cpg[bi + 1])
            else:
                ops.convT_1x2x2(cur, b["t_w"], b["t_b"], nxt)
            cur, flip = nxt, flip ^ 1
            H, W = 2 * H, 2 * W
            self.launches += 5 if fuse else 6  # fused: finalize + fold + 3 layers; else memset + 2 GroupNorm kernels + 3 layers
            self.launches += sum(c2 // 16 - 1 for r_ in (ra, rb) if r_ is not None)  # conv3d_rows: one kernel per 16 output channels
        return cur, names[flip]

    @torch.inference_mode()
    def segment_volume(self, features: torch.Tensor, want_probs: bool = True, want_logits: bool = True):
        """features: CUDA (C, D, h, w) fp16 or fp32 -> (logits, probs), each fp32 [D, 16h, 16w] (or None)."""
        cur, free = self._trunk(features)
        D, H, W, _ = cur.shape
        w_ = self._w
        scratch = self._buf(free, D * H * W * 8).view(D, H, W, 8)
        logits = torch.empty(D, H, W, device=self.device) if want_logits else None
        probs = torch.empty(D, H, W, device=self.device) if want_probs else None
        if W % 8 == 0 and self.rows8:  # always true downstream of the ViT (W = 16 w): one voxel per MMA row (conv_rows8.cu)
            ops.conv3d_rows8(cur, w_["o1_r8"], w_["o1_r8_b"], scratch)                    # output_layer.0 + GELU
            ops.conv3d_rows8_final(scratch, w_["o2_r8"], w_["o2_r8_b"], logits, probs)    # output_layer.2 + clip (+ sigmoid)
        elif W % 16 == 0:  # both on tensor cores, voxels packed into the MMA N (conv_wpack.cu; A/B arm: CVIT_HEAD_ROWS8=0)
            ops.conv3d_wpack8_gelu(cur, w_["o1_wp"], w_["o1_wp_b"], scratch)              # output_layer.0 + GELU
            ops.conv3d_wpack8_final(scratch, w_["o2_wp"], w_["o2_wp_b"], logits, probs)   # output_layer.2 + clip (+ sigmoid)
        else:
            ops.conv3d_halo(cur, w_["o1_img"], w_["o1_b16"], scratch, 1, 16)
            ops.head_out_conv(scratch, w_["o2_w"], w_["o2_b"], logits, probs)
        self.launches += 2
        return logits, probs

    @torch.inference_mode()
    def score_volume(self, features: torch.Tensor, labels: torch.Tensor, threshold: float = 0.5) -> torch.Tensor:
        """features: CUDA (C, D, h, w) fp16 or fp32, labels [D, 16h, 16w] (-1 = ignore) -> the eight masked sums of
        ``SegStats(probs, labels, threshold)`` over segment_volume's probabilities, fp64 [8] on the device.

        int8 labels (the caller guarantees values in {-1, 0, 1}) on planes whose width is a multiple of 8: output_layer.2
        scores inside its epilogue (``ops.conv3d_rows8_score``) and no probability volume is written. Other labels, or
        ``CVIT_HEAD_ROWS8=0``: segment_volume + seg_stats."""
        D, W = features.shape[1], 16 * features.shape[3]
        if labels.dtype != torch.int8 or W % 8 or not self.rows8:
            _, probs = self.segment_volume(features, want_logits=False)
            return ops.seg_stats(probs.reshape(-1), labels.to(self.device).reshape(-1).float().contiguous(), threshold)
        cur, free = self._trunk(features)
        D, H, W, _ = cur.shape
        w_ = self._w
        if tuple(labels.shape) != (D, H, W):
            raise CryovitB200Error(f"labels {tuple(labels.shape)} do not match the output volume {(D, H, W)}")
        scratch = self._buf(free, D * H * W * 8).view(D, H, W, 8)
        partials = self._buf("score_partials", ops.rows8_score_partials(D, H, W), torch.float64)
        out8 = torch.empty(8, device=self.device, dtype=torch.float64)
        ops.conv3d_rows8(cur, w_["o1_r8"], w_["o1_r8_b"], scratch)                                        # output_layer.0 + GELU
        ops.conv3d_rows8_score(scratch, w_["o2_r8"], w_["o2_r8_b"], labels.contiguous(), partials, out8, threshold)
        self.launches += 3  # + the finalize kernel
        return out8

    @torch.inference_mode()
    def forward_volume(self, x: torch.Tensor) -> torch.Tensor:
        """Reference signature (cryovit.py:36-40): x [B, C, D, h, w] -> clipped logits [B, 1, D, 16h, 16w]."""
        outs = [self.segment_volume(x[b].to(self.device), want_probs=False)[0] for b in range(x.shape[0])]
        return torch.stack(outs)[:, None]

    @torch.inference_mode()
    def forward(self, batch) -> torch.Tensor:
        """Reference signature (cryovit.py:42-49): batch.tomo_batch [B, D, C, h, w] -> probabilities [B, D, H, W]."""
        tb = batch.tomo_batch if hasattr(batch, "tomo_batch") else batch
        outs = [self.segment_volume(tb[b].to(self.device).permute(1, 0, 2, 3).contiguous(), want_logits=False)[1]
                for b in range(tb.shape[0])]
        return torch.stack(outs)

    __call__ = forward
