"""Cost of the deterministic mode of head training (trainer.deterministic) at the production crop: fp16 1536 x 128 x 32 x 32
features, 128 x 512 x 512 labels.

  python tools/determinism_probe.py --out DIR [--steps 30] [--reps 20]

* step time: a default and a deterministic trainer, each warmed up to its CUDA-graph replay, then --steps steps each,
  interleaved (default, deterministic, default, ...), each step timed with CUDA events around train_step;
* kernel time: every deterministic variant of the step against its atomic twin, at the step's shapes, --reps launches each
  between CUDA events (the variant's finalize included);
* scratch: the bytes of the deterministic trainer's scratch buffers after the steps.

The GPU's name and power limit are read in the same process. Writes DIR/determinism_probe.json and prints a markdown
summary."""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

DEV = "cuda"
BF16 = torch.bfloat16


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip().splitlines()[torch.cuda.current_device()]
            if q.returncode == 0 else f"unavailable ({q.stderr.strip()})"}


def crop(seed):
    g = torch.Generator().manual_seed(seed)
    f = torch.randn(1536, 128, 32, 32, generator=g).half().to(DEV)
    lab = (torch.rand(128, 512, 512, generator=g) < 0.3).float()
    lab[:, :64] = -1
    return f, lab.to(DEV)


def time_steps(args):
    from cryovit_b200.train import CryoVITHeadTrainerB200

    trs = {"default": CryoVITHeadTrainerB200(1536, seed=3), "deterministic": CryoVITHeadTrainerB200(1536, seed=3, deterministic=True)}
    f, lab = crop(1)
    for tr in trs.values():  # eager, eager, capture, then replays
        for _ in range(5):
            tr.train_step(f, lab)
    torch.cuda.synchronize()
    times = {k: [] for k in trs}
    for _ in range(args.steps):
        for k, tr in trs.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            tr.train_step(f, lab)
            b.record()
            b.synchronize()
            times[k].append(a.elapsed_time(b))
    det = trs["deterministic"]
    scratch = {k: v.numel() * v.element_size() for k, v in det._bufs.items() if k.startswith("det_scratch")}
    return times, scratch


def time_kernels(args):
    from cryovit_b200 import ops
    from cryovit_b200 import train_ops as T

    class Scratch:
        def __init__(self):
            self.b = {}

        def __call__(self, n, dtype=torch.float32):
            t = self.b.get(dtype)
            if t is None or t.numel() < n:
                t = self.b[dtype] = torch.empty(max(n, 1), device=DEV, dtype=dtype)
            return t

    r = lambda *s: torch.randn(*s, device=DEV).to(BF16)
    cases = {}
    for D, H, W, C, G in [(128, 32, 32, 1024, 128), (128, 64, 64, 128, 16), (128, 128, 128, 32, 8), (128, 256, 256, 32, 8)]:
        x, o, st = r(D, H, W, C), torch.empty(D, H, W, C, device=DEV, dtype=BF16), torch.empty(2 * G, device=DEV)
        gm, bt = torch.ones(C, device=DEV), torch.zeros(C, device=DEV)
        cases[f"groupnorm fwd {D}x{H}x{W}x{C}"] = lambda det, x=x, o=o, st=st, gm=gm, bt=bt, G=G: ops.groupnorm_ndhwc(x, o, gm, bt, st, G, 1e-3, det=det)
    p, lab = torch.rand(128 * 512 * 512, device=DEV), (torch.rand(128 * 512 * 512, device=DEV) < 0.3).float()
    cases["seg_stats 128x512x512"] = lambda det: ops.seg_stats(p, lab, det=det)
    for shp in [(128, 512, 512, 8), (128, 256, 256, 16)]:
        x, out = r(*shp), torch.zeros(shp[-1], device=DEV)
        cases[f"colsum {'x'.join(map(str, shp))}"] = lambda det, x=x, out=out: T.colsum(x, out, det=det)
    for shp in [(128, 32, 32, 192), (128, 256, 256, 16)]:
        da, z, dz, db = r(*shp), r(*shp), torch.empty(shp, device=DEV, dtype=BF16), torch.zeros(shp[-1], device=DEV)
        cases[f"gelu_bwd_colsum {'x'.join(map(str, shp))}"] = lambda det, da=da, z=z, dz=dz, db=db: T.gelu_bwd(da, z, dz, db, det=det)
    da, z = r(128, 512, 512, 8), r(128, 512, 512, 8)
    dzun, db = torch.empty(128, 256, 256, 32, device=DEV, dtype=BF16), torch.zeros(8, device=DEV)
    cases["gelu_bwd_unshuffle 128x512x512x8"] = lambda det: T.gelu_bwd_unshuffle(da, z, dzun, db, det=det)
    x, dy, zz = r(128, 64, 64, 128), r(128, 64, 64, 128), r(128, 64, 64, 128)
    dzb = torch.empty(128, 32, 32, 512, device=DEV, dtype=BF16)
    g1, g2, db1 = (torch.zeros(128, device=DEV) for _ in range(3))
    st1 = torch.ones(32, device=DEV)  # (sum, sum of squares) of the 16 groups: mean and variance of order 1 / N
    cases["groupnorm_bwd_gelu 128x64x64x128 (unshuffle)"] = lambda det: T.groupnorm_bwd_gelu(x, dy, dzb, torch.ones(128, device=DEV), st1, g1, g2, 16, 1e-3, zz, db1, True, det=det)
    for D, H, W, ci, co, dil in [(128, 512, 512, 8, 8, 1), (128, 256, 256, 32, 16, 2), (128, 256, 256, 16, 16, 1),
                                 (128, 128, 128, 32, 32, 8), (128, 32, 32, 1024, 192, 32), (128, 32, 32, 192, 192, 24),
                                 (128, 64, 64, 128, 64, 16), (128, 64, 64, 64, 64, 12)]:
        xx, dd = r(D, H, W, ci), r(D, H, W, co)
        cases[f"wgrad {D}x{H}x{W} {ci}->{co} dil {dil}"] = lambda det, xx=xx, dd=dd, dil=dil: T.conv_weight_gradient(xx, dd, dil, {}, det=det)
    R = 128 * 32 * 32
    xr, dr = r(R, 192), r(R, 512)
    cases["wgrad rows (convT 0) 192x512"] = lambda det: T.rows_weight_gradient(xr, dr, det=det)
    at, bt2, out = r(1024, R), r(1536, R), torch.zeros(1, 1024, 1536, device=DEV)
    koff = torch.zeros(1, dtype=torch.int32, device=DEV)
    cases["wgrad_splitk projection 1024x1536"] = lambda det: T.wgrad_splitk(at, bt2, out, koff, R, det=det)
    res = {}
    for name, fn in cases.items():
        row = {}
        for arm, det in (("atomic", None), ("deterministic", Scratch())):
            for _ in range(3):
                fn(det)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(args.reps):
                fn(det)
            b.record()
            b.synchronize()
            row[arm] = a.elapsed_time(b) / args.reps
        res[name] = row
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("determinism_probe: no CUDA device")
    from cryovit_b200 import build

    build.build()
    info = gpu_info()
    times, scratch = time_steps(args)
    kernels = time_kernels(args)
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    res = {"gpu": info, "step_ms": times, "scratch_bytes": scratch, "kernel_ms": kernels}
    (out / "determinism_probe.json").write_text(json.dumps(res, indent=1))
    print(f"GPU: {info['torch_name']} | nvidia-smi: {info['nvidia_smi']}")
    for k, v in times.items():
        print(f"step {k}: median {statistics.median(v):.3f} ms, min {min(v):.3f}, max {max(v):.3f} ({len(v)} graph-replayed steps)")
    print(f"scratch: {sum(scratch.values()) / 1e6:.1f} MB {scratch}")
    print("| kernel | atomic ms | deterministic ms | delta ms |\n|---|---|---|---|")
    for k, v in kernels.items():
        print(f"| {k} | {v['atomic']:.3f} | {v['deterministic']:.3f} | {v['deterministic'] - v['atomic']:+.3f} |")


if __name__ == "__main__":
    main()
