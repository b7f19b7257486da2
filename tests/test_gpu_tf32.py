"""The ``tf32`` operand mode on a B200: every ViT linear as a tcgen05 kind::tf32 MMA (the reference's own matmul
precision, run/dino_features.py:24), its producers (LayerNorm, GELU / SwiGLU epilogues, attention output, patches)
storing TF32-rounded fp32, and the model end to end against the fp32 oracle and the TF32 emulation of
tests/quant_emulation.py."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda"
ERR_UNSUPPORTED = -4
FMT_F16, FMT_OUT_F16, FMT_TF32, FMT_OUT_F32 = 1, 2, 4, 8


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def _tf32(t):
    from cryovit_b200.vit import round_tf32
    return round_tf32(t)


def _low_bits_zero(t, what):
    assert t.dtype == torch.float32
    bad = (t.contiguous().view(torch.int32) & 0x1FFF) != 0
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} stored values are not TF32 (13 low mantissa bits set)"


def _bound(a, w):
    """1e-5 of |a_i| |w_j| (Cauchy-Schwarz bound of each dot product): fp32 accumulation round-off over K; a
    descriptor or K-stepping mistake is an O(1) error against it."""
    return 1e-5 * a.double().norm(dim=1)[:, None] * w.double().norm(dim=1)[None, :]


def _assert_within(got, ref, tol, what):
    err = (got.double() - ref).abs()
    bad = int((err > tol).sum())
    assert bad == 0, f"{what}: {bad}/{err.numel()} outside tolerance, max abs err {err.max().item():.3e}"


@pytest.mark.parametrize("pair", [True, False])
@pytest.mark.parametrize("K", [256, 384, 1536, 4096])
def test_tf32_linears_vs_float64(cuda_lib, K, pair):
    """EPI_BIAS (bf16 out), EPI_BIAS_GELU and EPI_BIAS_SWIGLU (TF32-rounded fp32 out), EPI_SCALE_RESIDUAL (fp32) on
    TF32 operands, 2 x 1029 rows (ragged last tile), 256- and 128-wide N tiles, against a float64 matmul of the same
    TF32 values; the CTA-pair and single-CTA kernels agree bit for bit."""
    from cryovit_b200 import ops
    from cryovit_b200.vit import interleave_w12
    M = 2 * 1029
    a = _tf32(_rand(M, K, seed=1))
    b = _rand(1024, seed=3)
    prev = cuda_lib.cvit_set_gemm_pair(1 if pair else 0)
    gelu_out = {}
    try:
        for N in (1024, 384):
            w = _tf32(_rand(N, K, scale=K ** -0.5, seed=2))
            acc = a.double() @ w.double().t()
            tol = _bound(a, w)
            y = acc + b[:N].double()
            out = torch.full((M, N), float("nan"), device=DEV, dtype=torch.bfloat16)
            ops.linear_bias(a, w, b[:N], out)
            _assert_within(out, y, tol + y.abs() * 2.0 ** -8, f"tf32 linear_bias -> bf16 K={K} N={N}")
            outg = torch.full((M, N), float("nan"), device=DEV, dtype=torch.float32)
            ops.linear_bias(a, w, b[:N], outg, gelu=True)
            _low_bits_zero(outg, "GELU epilogue")
            g = F.gelu(y)
            # the epilogue's GELU: <= 2.6e-5 absolute, 2.1e-4 relative (ptx.cuh gelu_erf); then the TF32 rounding
            _assert_within(outg, g, 1.2 * tol + 3e-5 + g.abs() * (2.2e-4 + 2.0 ** -11), f"tf32 linear_bias+GELU -> fp32 K={K} N={N}")
            gelu_out[N] = outg
            x0 = _rand(M, N, seed=5)
            gam = _rand(N, seed=4)
            x = x0.clone()
            ops.linear_scale_residual(a, w, b[:N], gam, x)
            ref = x0.double() + gam.double() * y
            gy = (gam.double() * y).abs()
            _assert_within(x, ref, gam.double().abs() * tol + gy * 2.0 ** -22 + ref.abs() * 2.0 ** -23,
                           f"tf32 linear_scale_residual K={K} N={N}")
        w12 = _tf32(_rand(2048, K, scale=K ** -0.5, seed=6))
        b12 = _rand(2048, seed=7)
        w12i, b12i = interleave_w12(w12, b12)
        outs = torch.full((M, 1024), float("nan"), device=DEV, dtype=torch.float32)
        ops.linear_swiglu(a, w12i, b12i, outs)
        _low_bits_zero(outs, "SwiGLU epilogue")
        y12 = a.double() @ w12.double().t() + b12.double()
        tol12 = _bound(a, w12)
        s = F.silu(y12[:, :1024]) * y12[:, 1024:]
        # |d/dx1| <= 1.1 |x2|, |d/dx2| = |silu(x1)|: the accumulation bound through the product
        st = 1.1 * y12[:, 1024:].abs() * tol12[:, :1024] + F.silu(y12[:, :1024]).abs() * tol12[:, 1024:]
        _assert_within(outs, s, st + 1e-6 + s.abs() * (1e-5 + 2.0 ** -11), f"tf32 linear_swiglu -> fp32 K={K}")
    finally:
        cuda_lib.cvit_set_gemm_pair(prev)
    # the other kernel family (256-wide N tiles: CTA pair <-> single CTA) on the same inputs: same K order, same bits
    cuda_lib.cvit_set_gemm_pair(0 if pair else 1)
    try:
        w = _tf32(_rand(1024, K, scale=K ** -0.5, seed=2))
        o2 = torch.full((M, 1024), float("nan"), device=DEV, dtype=torch.float32)
        ops.linear_bias(a, w, b, o2, gelu=True)
        s2 = torch.full((M, 1024), float("nan"), device=DEV, dtype=torch.float32)
        ops.linear_swiglu(a, w12i, b12i, s2)
    finally:
        cuda_lib.cvit_set_gemm_pair(prev)
    assert torch.equal(o2, gelu_out[1024]) and torch.equal(s2, outs), "pair and single-CTA TF32 kernels differ"


@pytest.mark.parametrize("K,C", [(256, 1536), (640, 384), (256, 384)])
def test_tf32_patch_embed_vs_float64(cuda_lib, K, C):
    """EPI_PATCH_EMBED on TF32 patches / weights: K = 256 (one folded channel) and 640 (three channels)."""
    from cryovit_b200 import ops
    B, Np, T = 3, 343, 348
    patches = _tf32(torch.rand(B * Np, K, generator=torch.Generator().manual_seed(1)).to(DEV))
    w = _tf32(_rand(C, K, scale=K ** -0.5, seed=2))
    table = _rand(Np, C, seed=3)
    x = torch.full((B * T, C), 7.0, device=DEV)
    ops.patch_embed_gemm(patches, w, table, x, B, Np, T, 5)
    acc = (patches.double() @ w.double().t()).view(B, Np, C)
    ref = acc + table.double()
    got = x.view(B, T, C)
    _assert_within(got[:, 5:], ref, _bound(patches, w).view(B, Np, C) + acc.abs() * 2.0 ** -23 + ref.abs() * 2.0 ** -23,
                   f"tf32 patch embed K={K}")
    assert bool((got[:, :5] == 7.0).all()), "patch embed wrote outside the patch tokens"


@pytest.mark.parametrize("C", [384, 768, 1024, 1536])
def test_tf32_layernorm(cuda_lib, C):
    """The rounding LayerNorm stores exactly the TF32 rounding of what the fp32 LayerNorm stores."""
    from cryovit_b200 import ops
    M = 1031
    x = _rand(M, C, scale=3.0, seed=1) + 0.5
    g, b = _rand(C, seed=2), _rand(C, seed=3)
    o32 = torch.empty(M, C, device=DEV)
    ot = torch.full((M, C), float("nan"), device=DEV)
    ops.layernorm(x, g, b, o32, 1e-6)
    ops.layernorm(x, g, b, ot, 1e-6, tf32=True)
    _low_bits_zero(ot, "LayerNorm")
    assert torch.equal(ot, _tf32(o32))
    assert torch.allclose(o32, F.layer_norm(x, (C,), g, b, 1e-6), atol=1e-4, rtol=1e-4)


def test_tf32_patches(cuda_lib):
    """Both patchify paths in fp32: TF32 values, within half a TF32 step of the bicubic / copy reference, zero pad."""
    from cryovit_b200 import ops
    D, H, W = 3, 64, 96
    src = torch.randint(0, 256, (D, H, W), generator=torch.Generator().manual_seed(0), dtype=torch.uint8).to(DEV)
    OH, OW, ph, pw = ops.patch_grid(H, W)
    out = torch.full((D * ph * pw, 256), float("nan"), device=DEV)
    ops.preproc_patchify(src, out)
    _low_bits_zero(out, "u8 patchify")
    fp = F.pad(src.float()[:, None] / 255.0, (0, (W + 15) // 16 * 16 - W, 0, (H + 15) // 16 * 16 - H), mode="replicate")
    r = F.interpolate(fp, scale_factor=(14 / 16, 14 / 16), mode="bicubic")[:, 0]
    ref = r.view(D, ph, 14, pw, 14).permute(0, 1, 3, 2, 4).reshape(D * ph * pw, 196)
    assert torch.allclose(out[:, :196], ref, atol=1e-5, rtol=2.0 ** -10)
    assert bool((out[:, 196:] == 0).all())
    bf = torch.empty(D * ph * pw, 256, device=DEV, dtype=torch.bfloat16)
    ops.preproc_patchify(src, bf)
    assert (out[:, :196] - ref).abs().mean() < (bf[:, :196].float() - ref).abs().mean() / 4, "fp32 patches are not finer than bf16"
    x = _rand(2, 3, 56, 70, seed=1)
    o3 = torch.full((2 * 20, 640), float("nan"), device=DEV)
    ops.patchify_f32_3ch(x, o3)
    _low_bits_zero(o3, "3-channel patchify")
    ref3 = x.view(2, 3, 4, 14, 5, 14).permute(0, 2, 4, 1, 3, 5).reshape(40, 588)
    assert torch.equal(o3[:, :588], _tf32(ref3)) and bool((o3[:, 588:] == 0).all())


@pytest.mark.parametrize("B,T,H,scale", [(2, 1029, 3, 1.0), (3, 261, 2, 6.0), (16, 300, 8, 20.0)])
def test_tf32_attention_output(cuda_lib, B, T, H, scale):
    """bf16 q/k/v and probabilities, TF32-rounded fp32 output: within one fp16 ulp of the fp16-output kernel on the same
    q/k/v (TF32 and fp16 both keep 10 mantissa bits), and within the bf16 kernels' tolerance of fp32 SDPA."""
    from cryovit_b200 import ops
    C = H * 64
    qkv = (_rand(B * T, 3 * C, seed=1) * scale).bfloat16()
    o32 = torch.full((B * T, C), float("nan"), device=DEV)
    o16 = torch.full((B * T, C), float("nan"), device=DEV, dtype=torch.float16)
    ops.attention(qkv, o32, B, T, H)
    ops.attention(qkv, o16, B, T, H)
    _low_bits_zero(o32, "attention output")
    _, e = torch.frexp(o16.float())  # |v| in [2^(e-1), 2^e): one fp16 ulp is 2^(e-11), 2^-24 below the normal range
    ulp = torch.ldexp(torch.ones_like(o32), torch.clamp(e - 11, min=-24))
    assert bool(((o32 - o16.float()).abs() <= ulp).all()), "fp32 attention output is more than one fp16 ulp from the fp16 one"
    q, k, v = qkv.float().view(B, T, 3, H, 64).permute(2, 0, 3, 1, 4)
    ref = F.scaled_dot_product_attention(q, k, v).permute(0, 2, 1, 3).reshape(B * T, C)
    err = (o32 - ref).abs()
    assert bool((err <= 2e-2 * scale + 2e-2 * ref.abs()).all()), f"attention fp32 out vs SDPA: max err {err.max().item():.3e}"


def test_unsupported_format_flags_are_refused(cuda_lib):
    """Combinations without an instantiated kernel return CVIT_ERR_UNSUPPORTED with a message; none runs in another
    format. The torch front end refuses mixed operand types before the library sees them."""
    from cryovit_b200 import ops
    from cryovit_b200._lib import CryovitB200Error
    lib = cuda_lib
    M, N, K = 256, 256, 256
    a, w, b = torch.zeros(M, K, device=DEV), torch.zeros(N, K, device=DEV), torch.zeros(N, device=DEV)
    out, x = torch.zeros(M, N, device=DEV), torch.zeros(M, N, device=DEV)
    P = lambda t: t.data_ptr()  # noqa: E731
    for gelu, fmt in [(0, FMT_TF32 | FMT_F16), (0, FMT_OUT_F32), (1, FMT_OUT_F32), (1, FMT_TF32), (0, FMT_TF32 | FMT_OUT_F32),
                      (1, FMT_TF32 | FMT_OUT_F32 | FMT_OUT_F16), (1, FMT_F16 | FMT_OUT_F32)]:
        rc = lib.cvit_linear_bias_fmt(P(a), K, P(w), P(b), P(out), N, M, N, K, gelu, fmt, None)
        assert rc == ERR_UNSUPPORTED, (gelu, fmt, rc)
        assert b"not instantiated" in lib.cvit_last_error()
    for fmt in (FMT_TF32, FMT_OUT_F32, FMT_TF32 | FMT_F16 | FMT_OUT_F32):
        assert lib.cvit_linear_swiglu_fmt(P(a), K, P(w), P(b), P(out), N // 2, M, N, K, fmt, None) == ERR_UNSUPPORTED, fmt
    for fmt in (FMT_TF32 | FMT_F16, FMT_OUT_F32, FMT_TF32 | FMT_OUT_F32):
        assert lib.cvit_linear_scale_residual_fmt(P(a), K, P(w), P(b), P(b), P(x), N, M, N, K, fmt, None) == ERR_UNSUPPORTED, fmt
    for fmt in (FMT_TF32, FMT_OUT_F32 | FMT_F16, FMT_OUT_F32 | FMT_OUT_F16, FMT_F16):
        assert lib.cvit_attention_fwd_fmt(P(a), P(out), 1, 128, 1, 64, fmt, None) == ERR_UNSUPPORTED, fmt
        assert b"unsupported format" in lib.cvit_last_error()
    for fmt in (FMT_F16, FMT_OUT_F32, FMT_TF32 | FMT_OUT_F32):
        assert lib.cvit_patch_embed_gemm_fmt(P(a), K, P(w), P(b), P(x), N, 1, M, M, 0, N, K, fmt, None) == ERR_UNSUPPORTED, fmt
    with pytest.raises(CryovitB200Error):
        ops.linear_bias(a, w.bfloat16(), b, out.bfloat16())
    with pytest.raises(CryovitB200Error):
        ops.linear_bias(a.bfloat16(), w.bfloat16(), b, out)  # fp32 output from 16-bit operands
    with pytest.raises(CryovitB200Error):
        ops.layernorm(x, b, b, out.bfloat16(), 1e-6, tf32=True)


# ------------------------------------------------------------------------------------------------- end to end
def _errs(got, ref):
    got, ref = got.double().reshape(-1, got.shape[-1]), ref.double().reshape(-1, ref.shape[-1])
    rel = (got - ref).norm(dim=-1) / ref.norm(dim=-1)
    return rel.max().item(), rel.mean().item()


def test_tf32_vits_vs_oracle_and_golden(cuda_lib):
    """ViT-S (12 blocks) in tf32 mode against the fp32 oracle and the transformers golden: 4x inside the 1e-2 tolerance
    every 16-bit mode is held to."""
    from cryovit_b200.vit import CONFIGS, DinoVisionTransformerB200, random_state_dict
    from oracle import dinov2 as odino
    from pathlib import Path

    cfg = CONFIGS["dinov2_vits14_reg"]
    sd = random_state_dict(cfg, seed=0)
    x = torch.rand(2, 3, 392, 392, generator=torch.Generator().manual_seed(1))
    model = DinoVisionTransformerB200(cfg, "tf32").load_state_dict(sd).cuda()
    out = model.forward_features(x.cuda())
    got = out["x_norm_patchtokens"].float().cpu()
    ref = odino.forward_features(sd, x, cfg.num_heads)
    rmax, rmean = _errs(got, ref["x_norm_patchtokens"])
    print(f"\n[tf32] ViT-S vs oracle: max {rmax:.3e} mean {rmean:.3e}")
    assert rmax <= 2.5e-3
    assert _errs(out["x_norm_clstoken"].float().cpu()[:, None], ref["x_norm_clstoken"][:, None])[0] <= 2.5e-3
    hf = np.load(Path(__file__).resolve().parent / "golden" / "dinov2_hf.npz")
    gmax, _ = _errs(got[:, ::7], torch.from_numpy(hf["dinov2_vits_hf_patchtokens"]))
    print(f"[tf32] ViT-S vs transformers golden: max {gmax:.3e}")
    assert gmax <= 2.5e-3


@pytest.mark.parametrize("dim,heads,ffn,hidden", [(768, 12, "mlp", 3072), (1024, 16, "mlp", 4096), (1536, 24, "swiglu", 4096)])
def test_tf32_every_width_vs_oracle(cuda_lib, dim, heads, ffn, hidden):
    from cryovit_b200.vit import DinoVisionTransformerB200, ViTConfig, random_state_dict
    from oracle import dinov2 as odino

    cfg = ViTConfig(f"w{dim}", dim, 3, heads, ffn, hidden)
    sd = random_state_dict(cfg, seed=2)
    x = torch.rand(3, 3, 56, 84, generator=torch.Generator().manual_seed(3))
    model = DinoVisionTransformerB200(cfg, "tf32").load_state_dict(sd).cuda()
    got = model.forward_features(x.cuda())["x_norm_patchtokens"].float().cpu()
    ref = odino.forward_features(sd, x, cfg.num_heads)["x_norm_patchtokens"]
    rmax, rmean = _errs(got, ref)
    print(f"\n[tf32] width {dim} ({ffn}) vs oracle: max {rmax:.3e} mean {rmean:.3e}")
    assert rmax <= 2.5e-3


@pytest.mark.parametrize("case", ["seed 0", "heavy-tailed x10", "heavy-tailed x50"])
def test_tf32_vitg_one_slice_tracks_reference_arithmetic(cuda_lib, case):
    """ViT-g/14-reg4 (40 blocks) on one 448 x 448 slice against the fp32 oracle, next to the reference's own TF32
    arithmetic emulated on the same weights (quant_emulation.forward_emulated(..., "T", "T", "T")). Random init: mean and
    worst token <= 1.5x the emulation; heavy-tailed (trained-like, ill-conditioned at x50) weights: <= 2x."""
    from cryovit_b200.vit import CONFIGS, DinoVisionTransformerB200, random_state_dict
    from test_gpu_parity import _oracle_fp32_on_gpu, _tf32_emulation_on_gpu, heavy_tailed_state_dict

    cfg = CONFIGS["dinov2_vitg14_reg"]
    sd = random_state_dict(cfg, seed=0) if case == "seed 0" else heavy_tailed_state_dict(cfg, 21, 10.0 if "x10" in case else 50.0)
    x = torch.rand(1, 3, 448, 448, generator=torch.Generator().manual_seed(1))
    model = DinoVisionTransformerB200(cfg, "tf32").load_state_dict(sd).cuda()
    got = model.forward_features(x.cuda())["x_norm_patchtokens"].float().cpu()
    del model
    torch.cuda.empty_cache()
    sdg = {k: v.cuda() for k, v in sd.items()}
    ref = _oracle_fp32_on_gpu(sdg, x, cfg.num_heads)
    emu = _tf32_emulation_on_gpu(sdg, x, cfg.num_heads)
    del sdg
    torch.cuda.empty_cache()
    (gmax, gmean), (emax, emean) = _errs(got, ref), _errs(emu, ref)
    print(f"\n[tf32] ViT-g {case}: max {gmax:.3e} mean {gmean:.3e}; TF32 emulation max {emax:.3e} mean {emean:.3e}")
    k = 1.5 if case == "seed 0" else 2.0
    assert gmean <= k * emean and gmax <= k * emax


def test_tf32_vitg_full_size_tomogram(cuda_lib):
    """One 128 x 512 x 512 u8 tomogram at slice batch 128: finite, bit-identical to slice batch 48, and 16 of its slices
    within 2e-3 (worst token) of the fp32 oracle evaluated on the GPU."""
    from cryovit_b200.extract import extract_tomogram
    from cryovit_b200.vit import CONFIGS, DinoVisionTransformerB200, random_state_dict
    from oracle import preproc as opre
    from test_gpu_parity import _oracle_fp32_on_gpu

    cfg = CONFIGS["dinov2_vitg14_reg"]
    sd = random_state_dict(cfg, seed=0)
    model = DinoVisionTransformerB200(cfg, "tf32").load_state_dict(sd).cuda()
    tomo = np.random.default_rng(5).integers(0, 256, size=(128, 512, 512), dtype=np.uint8)
    full = extract_tomogram(tomo, model, batch_size=128)
    assert full.shape == (1536, 128, 32, 32) and full.dtype == np.float16 and np.isfinite(full).all()
    ragged = extract_tomogram(tomo, model, batch_size=48)
    assert np.array_equal(full, ragged), "features depend on the slice batch size"
    del model, ragged
    torch.cuda.empty_cache()
    ks = list(range(3, 128, 8))
    x = opre.dino_transform(opre.load_tomogram(tomo[ks]))
    sdg = {k: v.cuda() for k, v in sd.items()}
    ref = _oracle_fp32_on_gpu(sdg, x, cfg.num_heads).half().float()
    del sdg
    torch.cuda.empty_cache()
    got = torch.from_numpy(full[:, ks].astype(np.float32)).reshape(1536, len(ks), 1024).permute(1, 2, 0)
    rmax, rmean = _errs(got, ref)
    print(f"\n[tf32] full-size run, 16 slices vs oracle: max {rmax:.3e} mean {rmean:.3e}")
    assert rmax <= 2e-3


def test_tf32_through_the_entry_point(cuda_lib, tmp_path, monkeypatch):
    """CRYOVIT_B200_OPERANDS=tf32 reaches python -m cryovit.training.dino_features without a config key: the result file
    round-trips and its features are closer to the oracle than the default mode's."""
    from cryovit.training.dino_features import main
    from cryovit_b200.host import hdf
    from cryovit_b200.vit import CONFIGS, build_model, random_state_dict
    from oracle import dinov2 as odino
    from oracle import extract as oextract
    from oracle import preproc as opre

    monkeypatch.setenv("CRYOVIT_B200_OPERANDS", "tf32")
    assert build_model("dinov2_vits14_reg").operands == "tf32"
    monkeypatch.delenv("CRYOVIT_B200_OPERANDS")
    assert build_model("dinov2_vits14_reg").operands == "mixed-attn"
    cfg = CONFIGS["dinov2_vits14_reg"]
    sd = random_state_dict(cfg, seed=4)
    data = np.random.default_rng(9).integers(0, 256, (5, 64, 96), dtype=np.uint8)
    want = oextract.dino_features(opre.dino_transform(opre.load_tomogram(data)), odino.OracleDino(sd, cfg.num_heads), 2)
    errs = {}
    for mode in ("tf32", None):
        root = tmp_path / (mode or "default")
        hdf.write_tomogram(root / "dino_features" / "Q18" / "a.hdf", {"data": data})
        ckpt = root / "models" / "DINOv2" / "checkpoints" / "dinov2_vits14_reg4_pretrain.pth"
        ckpt.parent.mkdir(parents=True)
        torch.save(sd, ckpt)
        if mode:
            monkeypatch.setenv("CRYOVIT_B200_OPERANDS", mode)
        else:
            monkeypatch.delenv("CRYOVIT_B200_OPERANDS", raising=False)
        main([f"paths.data_dir={root}", f"paths.exp_dir={root}/exp", f"paths.model_dir={root}/models", "sample=Q18",
              "batch_size=2", "+dino_variant=dinov2_vits14_reg"])
        out = hdf.read_tomogram(root / "tomograms" / "Q18" / "a.hdf")
        assert np.array_equal(out["data"], data)
        got = out["dino_features"]
        assert got.dtype == np.float16 and got.shape == want.shape
        g, w = torch.from_numpy(got.astype(np.float32)), torch.from_numpy(want.astype(np.float32))
        rel = (g - w).norm(dim=0) / w.norm(dim=0)
        errs[mode or "default"] = (rel.max().item(), rel.mean().item())
    print(f"\n[tf32] entry point vs oracle (max, mean): {errs}")
    assert errs["tf32"][0] <= 1e-2 and errs["tf32"][1] < errs["default"][1]
