"""Batch training step of the CryoVIT head at BASELINE config 5's crop (features (1536, 128, 32, 32) fp16, labels
(128, 512, 512)): for batch sizes 1, 2, 4 and 8, the graph-replayed step time (``train_batch``: forward + backward from
its CUDA graph, all-reduce no-op on one GPU, AdamW), per step and per crop, and the peak allocated memory of a fresh
trainer; B = 1 also through ``train_step``, the fit loop's single-crop path. Then the cost of summing one sample's
gradient bucket into the step's (``cvit_accumulate_f32`` over 8.4 M fp32 numbers), the work a batch adds per extra crop.
The card's name and power limit are read in the same run.

    python tools/train_batch_probe.py [steps]     (default 20 timed steps per batch size)"""
import json
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from cryovit_b200 import build  # noqa: E402
from cryovit_b200 import train_ops as T  # noqa: E402
from cryovit_b200.train import CryoVITHeadTrainerB200  # noqa: E402

build.build()
STEPS = int(sys.argv[1]) if len(sys.argv) > 1 else 20
C, D, h, w = 1536, 128, 32, 32


def crop(seed: int):
    g = torch.Generator(device="cuda").manual_seed(seed)
    f = (torch.randn(C, D, h, w, generator=g, device="cuda") * 0.5).half()
    lab = (torch.rand(D, 16 * h, 16 * w, generator=g, device="cuda") < 0.1).float()
    lab[::5] = -1
    return f, lab


def timed(step, n: int) -> list[float]:
    out = []
    for _ in range(n):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        step()
        e.record()
        torch.cuda.synchronize()
        out.append(s.elapsed_time(e))
    return out


def median(xs):
    return sorted(xs)[len(xs) // 2]


def run(B: int, single: bool) -> dict:
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    crops = [crop(s) for s in range(B)]
    tr = CryoVITHeadTrainerB200(C, seed=0)
    step = (lambda: tr.train_step(*crops[0])) if single else (lambda: tr.train_batch(crops))
    timed(step, 4)  # two eager steps, the capture (+ its replay), one replay
    assert any("graph" in e for e in tr._graphs.values()), "the step was not captured"
    ts = timed(step, STEPS)
    peak = (torch.cuda.max_memory_allocated() - base) / 1e9
    ms = median(ts)
    row = {"B": B, "path": "train_step" if single else "train_batch", "ms_per_step": round(ms, 3), "ms_per_crop": round(ms / B, 3),
           "min_ms": round(min(ts), 3), "max_ms": round(max(ts), 3), "peak_allocated_GB": round(peak, 2),
           "sample_bytes_GB": round(tr.sample_bytes(D, h, w) / 1e9, 2)}
    del tr, crops, step
    return row


def accumulate_cost() -> dict:
    tr = CryoVITHeadTrainerB200(C, seed=0)
    src = torch.randn_like(tr.flat_g)
    T.accumulate(tr.flat_g, src)
    n = 200
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n):
        T.accumulate(tr.flat_g, src)
    e.record()
    torch.cuda.synchronize()
    us = s.elapsed_time(e) / n * 1e3
    return {"elements": tr.flat_g.numel(), "us_per_call": round(us, 2), "GB_per_s": round(3 * 4 * tr.flat_g.numel() / us / 1e3, 1)}


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
card = {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else smi.stderr.strip()}
print("card:", card)
rows = [run(1, True)] + [run(B, False) for B in (1, 2, 4, 8)]
for r in rows:
    print(f"B={r['B']} {r['path']:11s} {r['ms_per_step']:8.2f} ms/step {r['ms_per_crop']:7.2f} ms/crop (min {r['min_ms']:.2f} max {r['max_ms']:.2f}) "
          f"peak {r['peak_allocated_GB']:6.2f} GB (sample_bytes {r['sample_bytes_GB']:.2f} GB)")
acc = accumulate_cost()
print(f"gradient accumulation: {acc['us_per_call']:.1f} us per extra crop over {acc['elements']} fp32 ({acc['GB_per_s']} GB/s)")
print(json.dumps({"card": card, "crop": [C, D, h, w], "timed_steps": STEPS, "rows": rows, "accumulate": acc}))
