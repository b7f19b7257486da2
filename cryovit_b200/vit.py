"""B200-native DINOv2 (with registers) feature extractor: the object the reference obtains from
``torch.hub.load("facebookresearch/dinov2", "dinov2_vitg14_reg")`` (reference run/dino_features.py:25-28,336).

It mirrors what the reference uses of that object -- ``.cuda()``, ``.eval()``, ``forward_features(x)`` returning
``{"x_norm_patchtokens": ...}`` (run/dino_features.py:58) -- and accepts a state dict with the upstream
parameter names (``patch_embed.proj.weight``, ``blocks.<i>.attn.qkv.weight``, ``blocks.<i>.mlp.w12.weight`` ...),
so a downloaded DINOv2 checkpoint loads unchanged. All arithmetic of the forward pass runs in the sm_100a
kernels behind the C ABI (``cryovit_b200.ops``); torch only owns the device buffers.

Layout in HBM for a batch of B slices (T tokens per slice, C channels, F hidden):
    patches  bf16 [B*Np, Kp]      im2col rows of the 14x14 patches (one channel, Kp = 256; or 3 channels, 640)
    x        fp32 [B*T, C]        residual stream (kept fp32: 40 blocks of 16-bit updates accumulate in fp32)
    ln       op16 [B*T, C]        LayerNorm output feeding qkv / FFN GEMMs
    qkv      op16 [B*T, 3C]       (token, {q,k,v}, head, 64)
    attn     op16 [B*T, C]
    hidden   bf16 [B*T, F]        post-activation FFN hidden
    features fp16 [C, D, Np]      the reference's on-disk layout (C, D, h, w)

``operands="tf32"`` runs every linear (patch embedding, qkv, proj, w12 / fc1, w3 / fc2) as a tcgen05 kind::tf32 MMA,
the reference's own matmul precision (run/dino_features.py:24 ``set_float32_matmul_precision("high")``): patches, ln,
attn and hidden are fp32 holding TF32-rounded values, and so are the weights (rounded once when packed); q/k/v and the
softmax probabilities stay bf16 (the emulation in tests/quant_emulation.py shows their format does not move the
end-to-end error). The FFN hidden activations and w3 / fc2, where DINOv2's large-magnitude channels are born, get 10
mantissa bits at fp32 range, so the error tracks the reference's own arithmetic on ill-conditioned (trained-like)
weights too, at half the tensor-core rate of the 16-bit modes. The features are written as fp16 in every mode.

op16 = the operand format of the 16-bit modes, chosen by ``operands`` (``"mixed-attn"`` default | ``"mixed"`` | ``"fp16"`` | ``"bf16"``). The reference runs
these GEMMs in TF32 (10 mantissa bits). ln and the attention output are bounded (LayerNorm output times gamma; convex
combinations of v), so ``mixed`` / ``fp16`` give them and the weights they meet (qkv, proj, w12 / fc1) the same 10 bits
as IEEE fp16 at the same bytes (bf16 has 7); the FFN hidden activations, where DINOv2's large-magnitude channels are
born, and the w3 / fc2 weights they meet stay bf16 (fp32 range) in every mode. ``mixed`` keeps q/k/v and the softmax
probabilities bf16: emulating each rounding inside the fp32 oracle (tests/quant_emulation.py, ViT-g, 40 blocks,
LayerScale 1.0) shows that their format does not move the end-to-end error at all (fp16 everywhere 4.10e-3; fp16 with
bf16 q/k/v/P 4.10e-3; bf16 everywhere 8.83e-3; only LayerNorm-side fp16 6.39e-3), while bf16 probabilities cannot
overflow whatever running maximum the flash softmax uses. Measured on B200, ViT-g random init with LayerScale 1.0 (the
worst case): per-token relative error 8.8e-3 (bf16) -> 4.1e-3 (fp16 / mixed) against the 1e-2 tolerance. bf16 operands
are ~4 % faster under the 1000 W power cap (the tensor cores draw more multiplying 11-bit significands) but leave a 12 %
margin only. ``mixed-attn`` (the default, and the format the benchmark reports) is ``mixed`` with the FFN input side --
norm2 output and the w12 / fc1 weights, 44 % of the FLOPs -- left in bf16: measured on one box, interleaved
(tools/operands_probe.py, three weight sets x 4 slices): mixed 4.1-4.4e-3 at 390-392 slices/s, mixed-attn 5.6-5.8e-3 at
401 slices/s, bf16 8.2-9.0e-3 at 405 slices/s. The bar is the worst token of the parity sweep <= 8e-3 (the 1e-2 tolerance
with 20 % to spare, tests/test_gpu_parity.py::test_vitg_parity_sweep): mixed-attn keeps 28 % under that bar and gets
back 2.5 of the 3.5 % that full fp16 significands cost; ``mixed`` stays one switch away for twice the margin.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch
import torch.nn.functional as F

from . import nvtx, ops
from ._lib import CryovitB200Error


@dataclass(frozen=True)
class ViTConfig:
    name: str
    embed_dim: int
    depth: int
    num_heads: int
    ffn: str  # "mlp" (fc1-GELU-fc2) or "swiglu" (w12 / w3)
    hidden: int
    num_register_tokens: int = 4
    patch_size: int = 14
    pos_grid: int = 37  # 518 / 14, the pre-training grid
    ln_eps: float = 1e-6
    init_values: float = 1.0  # LayerScale init used by the hub constructors


def _swiglu_hidden(dim: int) -> int:
    # upstream SwiGLUFFNFused: hidden = (int(4*dim * 2/3) + 7) // 8 * 8
    return (int(4 * dim * 2 / 3) + 7) // 8 * 8


OPERAND_MODES = ("mixed-attn", "mixed", "fp16", "bf16", "tf32")
DEFAULT_OPERANDS = "mixed-attn"

CONFIGS = {
    "dinov2_vits14_reg": ViTConfig("dinov2_vits14_reg", 384, 12, 6, "mlp", 1536),
    "dinov2_vitb14_reg": ViTConfig("dinov2_vitb14_reg", 768, 12, 12, "mlp", 3072),
    "dinov2_vitl14_reg": ViTConfig("dinov2_vitl14_reg", 1024, 24, 16, "mlp", 4096),
    "dinov2_vitg14_reg": ViTConfig("dinov2_vitg14_reg", 1536, 40, 24, "swiglu", _swiglu_hidden(1536)),
}


def random_state_dict(cfg: ViTConfig, seed: int = 0) -> dict[str, torch.Tensor]:
    """Seeded random-init parameters under the upstream key names (fp32, CPU). LayerScale gamma = init_values
    (1.0): the worst case for error accumulation. Used by tests / bench, where no checkpoint can be fetched."""
    g = torch.Generator().manual_seed(seed)
    C, Fh = cfg.embed_dim, cfg.hidden

    def tn(*shape, std=0.02):
        return torch.randn(*shape, generator=g) * std

    sd = {
        "cls_token": tn(1, 1, C, std=1e-6),
        "pos_embed": tn(1, 1 + cfg.pos_grid**2, C),
        "register_tokens": tn(1, cfg.num_register_tokens, C, std=1e-6),
        "mask_token": torch.zeros(1, C),
        "patch_embed.proj.weight": tn(C, 3, cfg.patch_size, cfg.patch_size, std=(3 * cfg.patch_size**2) ** -0.5),
        "patch_embed.proj.bias": tn(C),
        "norm.weight": 1.0 + tn(C),
        "norm.bias": tn(C),
    }
    for i in range(cfg.depth):
        p = f"blocks.{i}."
        sd[p + "norm1.weight"] = 1.0 + tn(C)
        sd[p + "norm1.bias"] = tn(C)
        sd[p + "attn.qkv.weight"] = tn(3 * C, C, std=C**-0.5)
        sd[p + "attn.qkv.bias"] = tn(3 * C)
        sd[p + "attn.proj.weight"] = tn(C, C, std=C**-0.5)
        sd[p + "attn.proj.bias"] = tn(C)
        sd[p + "ls1.gamma"] = torch.full((C,), cfg.init_values)
        sd[p + "norm2.weight"] = 1.0 + tn(C)
        sd[p + "norm2.bias"] = tn(C)
        if cfg.ffn == "swiglu":
            sd[p + "mlp.w12.weight"] = tn(2 * Fh, C, std=C**-0.5)
            sd[p + "mlp.w12.bias"] = tn(2 * Fh)
            sd[p + "mlp.w3.weight"] = tn(C, Fh, std=Fh**-0.5)
            sd[p + "mlp.w3.bias"] = tn(C)
        else:
            sd[p + "mlp.fc1.weight"] = tn(Fh, C, std=C**-0.5)
            sd[p + "mlp.fc1.bias"] = tn(Fh)
            sd[p + "mlp.fc2.weight"] = tn(C, Fh, std=Fh**-0.5)
            sd[p + "mlp.fc2.bias"] = tn(C)
        sd[p + "ls2.gamma"] = torch.full((C,), cfg.init_values)
    return sd


def interleave_w12(w12: torch.Tensor, b12: torch.Tensor, tile: int = 256):
    """Re-order SwiGLU w12 rows so each ``tile``-row block is [tile/2 rows of w1 | the matching rows of w2];
    the GEMM epilogue then finds silu-input and gate of the same hidden unit in one accumulator tile."""
    two_f = w12.shape[0]
    Fh, half = two_f // 2, tile // 2
    if Fh % half:
        raise CryovitB200Error(f"SwiGLU hidden size {Fh} must be a multiple of {half}")
    idx = torch.arange(Fh, device=w12.device).view(-1, half)
    perm = torch.cat([idx, idx + Fh], dim=1).reshape(-1)
    return w12[perm].contiguous(), b12[perm].contiguous()


def interpolate_pos_embed(pos_embed: torch.Tensor, gh: int, gw: int, pos_grid: int) -> torch.Tensor:
    """Upstream interpolate_pos_encoding for the *_reg models (interpolate_offset=0.0, antialias=True;
    HF:93-145): bicubic, antialiased resample of the pos_grid^2 patch table to (gh, gw). fp32, returns
    (cls_pos [C], patch_pos [gh*gw, C]). Parameter preparation, done once per grid size."""
    pe = pos_embed.float()
    cls_pos, patch_pos = pe[0, 0], pe[0, 1:]
    C = patch_pos.shape[-1]
    if (gh, gw) != (pos_grid, pos_grid):
        patch_pos = patch_pos.reshape(1, pos_grid, pos_grid, C).permute(0, 3, 1, 2)
        patch_pos = F.interpolate(patch_pos, size=(gh, gw), mode="bicubic", antialias=True, align_corners=False)
        patch_pos = patch_pos.permute(0, 2, 3, 1).reshape(gh * gw, C)
    return cls_pos.contiguous(), patch_pos.contiguous()


class DinoVisionTransformerB200:
    """Inference-only DINOv2-reg ViT on one B200. Not an nn.Module: weights live as pre-packed device buffers."""

    KP1 = 256  # one-channel patch row, 196 -> 256
    KP3 = 640  # three-channel patch row, 588 -> 640

    def __init__(self, cfg: ViTConfig | str = "dinov2_vitg14_reg", operands: str | torch.dtype = DEFAULT_OPERANDS):
        self.cfg = CONFIGS[cfg] if isinstance(cfg, str) else cfg
        operands = {torch.float16: "fp16", torch.bfloat16: "bf16"}.get(operands, operands)
        if operands not in OPERAND_MODES:
            raise CryovitB200Error(f"operands must be one of {OPERAND_MODES} (or torch.float16 / torch.bfloat16), got {operands!r}")
        self.operands = operands
        self.tf32 = operands == "tf32"
        # ln / attention output / qkv, proj, w12 weights  |  q, k, v and the softmax probabilities
        self.operand_dtype = torch.float32 if self.tf32 else torch.bfloat16 if operands == "bf16" else torch.float16
        self.qkv_dtype = torch.float16 if operands == "fp16" else torch.bfloat16
        # norm2 output and the w12 / fc1 weights it meets: "mixed-attn" keeps the FFN (44 % of the FLOPs) all-bf16
        self.ffn_dtype = self.operand_dtype if operands in ("tf32", "mixed", "fp16") else torch.bfloat16
        # patches, FFN hidden activations and the patch-embed / w3 / fc2 weights: bf16 in every 16-bit mode
        self.hidden_dtype = torch.float32 if self.tf32 else torch.bfloat16
        self.device: torch.device | None = None
        self._sd_cpu: dict[str, torch.Tensor] | None = None
        self._w: dict = {}
        self._pos_cache: dict = {}
        self._ws: dict = {}
        self.launches = 0  # kernels launched by this object (bench.py reports it)

    # ----------------------------------------------------------------------------- torch.hub-like surface
    @property
    def embed_dim(self) -> int:
        return self.cfg.embed_dim

    @property
    def patch_size(self) -> int:
        return self.cfg.patch_size

    @property
    def num_register_tokens(self) -> int:
        return self.cfg.num_register_tokens

    def load_state_dict(self, sd: dict[str, torch.Tensor], strict: bool = True):
        need = set(random_state_dict_keys(self.cfg))
        missing = sorted(need - set(sd))
        if strict and missing:
            raise CryovitB200Error(f"state dict is missing {len(missing)} keys, e.g. {missing[:3]}")
        self._sd_cpu = {k: v.detach().float().cpu() for k, v in sd.items()}
        if self.device is not None:
            self._pack()
        return self

    def state_dict(self) -> dict[str, torch.Tensor]:
        return dict(self._sd_cpu or {})

    def cuda(self, device=None):
        if not torch.cuda.is_available():
            raise CryovitB200Error("no CUDA device: the B200 hot path has no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        if self._sd_cpu is not None:
            self._pack()
        return self

    def to(self, device):
        d = torch.device(device)
        if d.type != "cuda":
            raise CryovitB200Error("DinoVisionTransformerB200 only runs on CUDA devices")
        return self.cuda(d.index)

    def eval(self):
        return self

    def __call__(self, x):
        return self.forward_features(x)["x_norm_clstoken"]

    # ----------------------------------------------------------------------------- weight packing
    def _pack(self) -> None:
        cfg, sd, dev = self.cfg, self._sd_cpu, self.device
        C = cfg.embed_dim
        f32 = lambda t: t.to(dev).float().contiguous()
        # weights of the bf16 side (patch embedding, w3 / fc2): TF32-rounded fp32 in tf32 mode
        bf = (lambda t: round_tf32(f32(t))) if self.tf32 else (lambda t: t.to(dev).to(torch.bfloat16).contiguous())
        if self.operand_dtype == torch.float16:
            def op(t):  # weights that meet an fp16 activation; fail loudly rather than store an inf
                if float(t.abs().max()) > 6.0e4:
                    raise CryovitB200Error("a weight exceeds the fp16 range: construct the model with operands='bf16' "
                                           "or operands='tf32'")
                return t.to(dev).to(torch.float16).contiguous()
        else:
            op = bf
        opf = op if self.ffn_dtype == self.operand_dtype else bf
        w = {}
        pw = sd["patch_embed.proj.weight"].float()  # [C, 3, 14, 14]
        w3 = torch.zeros(C, self.KP3)
        w3[:, :588] = pw.reshape(C, 588)
        w1 = torch.zeros(C, self.KP1)
        w1[:, :196] = pw.sum(dim=1).reshape(C, 196)  # the 3 input channels are identical copies
        w["pe_w3"], w["pe_w1"] = bf(w3), bf(w1)
        w["pe_bias"] = sd["patch_embed.proj.bias"].float()
        w["norm_w"], w["norm_b"] = f32(sd["norm.weight"]), f32(sd["norm.bias"])
        blocks = []
        for i in range(cfg.depth):
            p = f"blocks.{i}."
            b = {
                "n1w": f32(sd[p + "norm1.weight"]), "n1b": f32(sd[p + "norm1.bias"]),
                "qkv_w": op(sd[p + "attn.qkv.weight"]), "qkv_b": f32(sd[p + "attn.qkv.bias"]),
                "proj_w": op(sd[p + "attn.proj.weight"]), "proj_b": f32(sd[p + "attn.proj.bias"]),
                "ls1": f32(sd[p + "ls1.gamma"]), "ls2": f32(sd[p + "ls2.gamma"]),
                "n2w": f32(sd[p + "norm2.weight"]), "n2b": f32(sd[p + "norm2.bias"]),
            }
            if cfg.ffn == "swiglu":
                w12i, b12i = interleave_w12(sd[p + "mlp.w12.weight"].float(), sd[p + "mlp.w12.bias"].float())
                b["w12i"], b["b12i"] = opf(w12i), f32(b12i)
                b["out_w"], b["out_b"] = bf(sd[p + "mlp.w3.weight"]), f32(sd[p + "mlp.w3.bias"])
            else:
                b["fc1_w"], b["fc1_b"] = opf(sd[p + "mlp.fc1.weight"]), f32(sd[p + "mlp.fc1.bias"])
                b["out_w"], b["out_b"] = bf(sd[p + "mlp.fc2.weight"]), f32(sd[p + "mlp.fc2.bias"])
            blocks.append(b)
        w["blocks"] = blocks
        self._w = w
        self._pos_cache.clear()

    def _pos_tables(self, gh: int, gw: int):
        key = (gh, gw)
        if key not in self._pos_cache:
            sd, cfg = self._sd_cpu, self.cfg
            cls_pos, patch_pos = interpolate_pos_embed(sd["pos_embed"], gh, gw, cfg.pos_grid)
            table = (patch_pos + self._w["pe_bias"][None, :]).to(self.device).contiguous()
            special = torch.cat([sd["cls_token"].float()[0] + cls_pos[None, :], sd["register_tokens"].float()[0]], dim=0)
            self._pos_cache[key] = (table, special.to(self.device).contiguous())
        return self._pos_cache[key]

    def _workspace(self, B: int, T: int, Np: int, kp: int) -> dict:
        key = (B, T, Np, kp)
        if key not in self._ws:
            cfg, dev = self.cfg, self.device
            C, Fh, M = cfg.embed_dim, cfg.hidden, B * T
            hid = dict(device=dev, dtype=self.hidden_dtype)
            op16 = dict(device=dev, dtype=self.operand_dtype)
            self._ws = {  # keep one shape alive: a different batch shape replaces the buffers
                key: {
                    "patches": torch.empty(B * Np, kp, **hid),
                    "x": torch.empty(M, C, device=dev, dtype=torch.float32),
                    "ln": torch.empty(M, C, **op16),
                    "ln2": torch.empty(M if self.ffn_dtype != self.operand_dtype else 0, C, device=dev, dtype=self.ffn_dtype),
                    "qkv": torch.empty(M, 3 * C, device=dev, dtype=self.qkv_dtype),
                    "attn": torch.empty(M, C, **op16),
                    "hidden": torch.empty(M, Fh, **hid),
                }
            }
        return self._ws[key]

    # ----------------------------------------------------------------------------- forward
    def _require_ready(self):
        if self.device is None or not self._w:
            raise CryovitB200Error("model not ready: call load_state_dict(...) and .cuda() first")

    def _blocks(self, ws: dict, B: int, T: int) -> None:
        cfg = self.cfg
        x, ln, qkv, attn, hidden = ws["x"], ws["ln"], ws["qkv"], ws["attn"], ws["hidden"]
        ln2 = ws["ln2"] if self.ffn_dtype != self.operand_dtype else ln
        for i, b in enumerate(self._w["blocks"]):
            with nvtx.span(f"vit.block{i}.attn"):
                ops.layernorm(x, b["n1w"], b["n1b"], ln, cfg.ln_eps, tf32=self.tf32)
                ops.linear_bias(ln, b["qkv_w"], b["qkv_b"], qkv)
                ops.attention(qkv, attn, B, T, cfg.num_heads)
                ops.linear_scale_residual(attn, b["proj_w"], b["proj_b"], b["ls1"], x)
            with nvtx.span(f"vit.block{i}.ffn"):
                ops.layernorm(x, b["n2w"], b["n2b"], ln2, cfg.ln_eps, tf32=self.tf32)
                if cfg.ffn == "swiglu":
                    ops.linear_swiglu(ln2, b["w12i"], b["b12i"], hidden)
                else:
                    ops.linear_bias(ln2, b["fc1_w"], b["fc1_b"], hidden, gelu=True)
                ops.linear_scale_residual(hidden, b["out_w"], b["out_b"], b["ls2"], x)
        self.launches += 7 * len(self._w["blocks"])

    def _embed(self, ws: dict, B: int, T: int, gh: int, gw: int, pe_w: torch.Tensor) -> None:
        table, special = self._pos_tables(gh, gw)
        S = 1 + self.cfg.num_register_tokens
        ops.patch_embed_gemm(ws["patches"], pe_w, table, ws["x"], B, gh * gw, T, S)
        ops.assemble_special_tokens(ws["x"], special, B, T)
        self.launches += 2

    @torch.inference_mode()
    def forward_features(self, x: torch.Tensor) -> dict[str, torch.Tensor]:
        """Reference-facing entry (seam B2): x f32 [B, 3, H', W'] on the GPU, H', W' multiples of 14."""
        self._require_ready()
        if x.dim() != 4 or x.shape[1] != 3 or x.shape[2] % 14 or x.shape[3] % 14:
            raise CryovitB200Error(f"forward_features expects [B,3,H,W] with H,W multiples of 14, got {tuple(x.shape)}")
        x = x.to(self.device, torch.float32).contiguous()
        B, _, OH, OW = x.shape
        gh, gw = OH // 14, OW // 14
        S = 1 + self.cfg.num_register_tokens
        Np, T, C = gh * gw, gh * gw + S, self.cfg.embed_dim
        ws = self._workspace(B, T, Np, self.KP3)
        ops.patchify_f32_3ch(x, ws["patches"])
        self._embed(ws, B, T, gh, gw, self._w["pe_w3"])
        self._blocks(ws, B, T)
        xn = torch.empty(B * T, C, device=self.device, dtype=torch.float32)
        ops.layernorm(ws["x"], self._w["norm_w"], self._w["norm_b"], xn, self.cfg.ln_eps)
        self.launches += 2
        xn = xn.view(B, T, C)
        return {
            "x_norm_clstoken": xn[:, 0],
            "x_norm_regtokens": xn[:, 1:S],
            "x_norm_patchtokens": xn[:, S:],
            "x_prenorm": ws["x"].view(B, T, C),
            "masks": None,
        }

    @torch.inference_mode()
    def extract_into(self, slices: torch.Tensor, features: torch.Tensor, d0: int) -> None:
        """Fused path: raw slices (u8 or f32 in [0,1]) [B, H, W] on the GPU -> features[:, d0:d0+B] (fp16
        [C, D, gh, gw]). Pre-processing, ViT, final norm and the layout change all stay on the device."""
        self._require_ready()
        B, H, W = slices.shape
        _, _, gh, gw = ops.patch_grid(H, W)
        S = 1 + self.cfg.num_register_tokens
        Np, T = gh * gw, gh * gw + S
        if tuple(features.shape[2:]) != (gh, gw) or features.shape[0] != self.cfg.embed_dim:
            raise CryovitB200Error(f"features buffer {tuple(features.shape)} does not match (C,D,{gh},{gw})")
        ws = self._workspace(B, T, Np, self.KP1)
        ops.preproc_patchify(slices, ws["patches"])
        self._embed(ws, B, T, gh, gw, self._w["pe_w1"])
        self._blocks(ws, B, T)
        ops.final_norm_writeout(ws["x"], self._w["norm_w"], self._w["norm_b"], features.view(features.shape[0], features.shape[1], Np),
                                B, T, S, Np, d0, self.cfg.ln_eps)
        self.launches += 2

    @torch.inference_mode()
    def extract_preprocessed_into(self, data: torch.Tensor, features: torch.Tensor, d0: int) -> None:
        """Same as extract_into but from the reference's pre-processed input f32 [B, 3, H', W']."""
        self._require_ready()
        B, _, OH, OW = data.shape
        gh, gw = OH // 14, OW // 14
        S = 1 + self.cfg.num_register_tokens
        Np, T = gh * gw, gh * gw + S
        ws = self._workspace(B, T, Np, self.KP3)
        ops.patchify_f32_3ch(data.contiguous(), ws["patches"])
        self._embed(ws, B, T, gh, gw, self._w["pe_w3"])
        self._blocks(ws, B, T)
        ops.final_norm_writeout(ws["x"], self._w["norm_w"], self._w["norm_b"], features.view(features.shape[0], features.shape[1], Np),
                                B, T, S, Np, d0, self.cfg.ln_eps)
        self.launches += 2


def round_tf32(t: torch.Tensor) -> torch.Tensor:
    """fp32 -> the nearest TF32 value (8 exponent, 10 mantissa bits), ties away from zero, in fp32 with the 13 low
    mantissa bits zero: what cvt.rna.tf32.f32 gives for finite inputs. Non-finite values are refused."""
    t = t.float().contiguous()
    if not bool(torch.isfinite(t).all()):
        raise CryovitB200Error("round_tf32: the tensor holds inf or nan")
    return ((t.view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


def random_state_dict_keys(cfg: ViTConfig) -> list[str]:
    keys = ["cls_token", "pos_embed", "register_tokens", "patch_embed.proj.weight", "patch_embed.proj.bias",
            "norm.weight", "norm.bias"]
    per = ["norm1.weight", "norm1.bias", "attn.qkv.weight", "attn.qkv.bias", "attn.proj.weight", "attn.proj.bias",
           "ls1.gamma", "norm2.weight", "norm2.bias", "ls2.gamma"]
    per += ["mlp.w12.weight", "mlp.w12.bias", "mlp.w3.weight", "mlp.w3.bias"] if cfg.ffn == "swiglu" else \
           ["mlp.fc1.weight", "mlp.fc1.bias", "mlp.fc2.weight", "mlp.fc2.bias"]
    for i in range(cfg.depth):
        keys += [f"blocks.{i}.{k}" for k in per]
    return keys


def build_model(name: str = "dinov2_vitg14_reg", state_dict: dict | None = None, seed: int = 0,
                operands: str | torch.dtype | None = None) -> DinoVisionTransformerB200:
    """Stand-in for torch.hub.load(*dino_model): random-init (seeded) unless a state dict is given. ``operands``
    None reads CRYOVIT_B200_OPERANDS (``mixed-attn`` | ``mixed`` | ``fp16`` | ``bf16`` | ``tf32``, default mixed-attn), so the Hydra entry points can
    switch it without a config key the reference does not have."""
    if operands is None:
        import os

        operands = os.environ.get("CRYOVIT_B200_OPERANDS", DEFAULT_OPERANDS).lower()
        if operands not in OPERAND_MODES:
            raise CryovitB200Error(f"CRYOVIT_B200_OPERANDS must be one of {OPERAND_MODES}, got {operands!r}")
    m = DinoVisionTransformerB200(name, operands)
    m.load_state_dict(state_dict if state_dict is not None else random_state_dict(m.cfg, seed))
    return m
