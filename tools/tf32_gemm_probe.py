"""Time each ViT-g/14 linear alone on one GPU at slice batch 128 (M = 128 x 1029 tokens), in the tf32 operand mode
(tcgen05 kind::tf32) and in the default mixed-attn formats (kind::f16), with CUDA events over >= 0.5 s per GEMM after a
warm-up; prints TFLOP/s against the data-sheet dense peaks (1,125 TF32, 2,250 BF16/FP16), then the reference's own
TF32 path (bench.py's gpu_eager_baseline vit_tf32 leg) on the same GPU. The card's name and power limit are printed
first.  usage: python tools/tf32_gemm_probe.py"""
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from cryovit_b200 import ops  # noqa: E402
from cryovit_b200.vit import CONFIGS, interleave_w12, random_state_dict, round_tf32  # noqa: E402

PEAK = {"tf32": 1125.0, "16-bit": 2250.0}


def timed(fn, min_s=0.5):
    fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 1
    while True:
        s.record()
        for _ in range(reps):
            fn()
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e)
        if ms >= min_s * 1e3:
            return ms / reps
        reps = max(reps * 2, int(reps * min_s * 1.2e3 / max(ms, 1e-3)))


def main():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    print(f"gpu: {q}", flush=True)
    cfg = CONFIGS["dinov2_vitg14_reg"]
    C, Fh, M = cfg.embed_dim, cfg.hidden, 128 * 1029
    g = torch.Generator().manual_seed(0)
    dev = "cuda"
    # (name, N, K, kind): qkv EPI_BIAS, proj / w3 EPI_SCALE_RESIDUAL, w12 EPI_BIAS_SWIGLU
    shapes = [("qkv", 3 * C, C), ("proj", C, C), ("w12", 2 * Fh, C), ("w3", C, Fh)]
    x = torch.zeros(M, C, device=dev)
    gamma = torch.ones(C, device=dev)
    for mode in ("tf32", "16-bit"):
        for name, N, K in shapes:
            a32 = round_tf32(torch.randn(M, K, generator=g).to(dev))
            w32 = round_tf32((torch.randn(N, K, generator=g) * K ** -0.5).to(dev))
            bias = torch.zeros(N, device=dev)
            if mode == "tf32":
                a, w = a32, w32
            else:  # the default mixed-attn formats of the same linear
                dt = torch.float16 if name in ("qkv", "proj") else torch.bfloat16
                a, w = a32.to(dt), w32.to(dt)
            if name == "qkv":
                out = torch.empty(M, N, device=dev, dtype=torch.bfloat16 if mode == "tf32" else torch.float16)
                fn = lambda: ops.linear_bias(a, w, bias, out)  # noqa: E731
            elif name == "w12":
                wi, bi = interleave_w12(w, bias)
                out = torch.empty(M, N // 2, device=dev, dtype=torch.float32 if mode == "tf32" else torch.bfloat16)
                fn = lambda: ops.linear_swiglu(a, wi, bi, out)  # noqa: E731
            else:
                out = x
                fn = lambda: ops.linear_scale_residual(a, w, bias, gamma, x)  # noqa: E731
            ms = timed(fn)
            tf = 2.0 * M * N * K / ms / 1e9
            print(f"[{mode}] {name:5s} M={M} N={N} K={K}: {ms:.3f} ms  {tf:.0f} TFLOP/s  "
                  f"({100 * tf / PEAK[mode]:.0f} % of the {PEAK[mode]:.0f} TFLOP/s dense data-sheet figure)", flush=True)
            del a, w, a32, w32, out
            torch.cuda.empty_cache()
    import bench

    eager = bench.gpu_eager_baseline(torch, random_state_dict(cfg, seed=0))
    print(f"reference TF32 path (gpu_eager_baseline vit_tf32): {eager['vit_tf32']}", flush=True)


if __name__ == "__main__":
    main()
