#!/usr/bin/env python
"""What validation during head training costs, on full-size synthetic tomograms (1536 x 128 x 32 x 32 fp16 features,
int8 labels of 128 x 512 x 512):

  1. per tomogram: CryoVITHeadB200.score_volume (scoring inside the output convolution) against segment_volume + the
     int8 -> fp32 label conversion + seg_stats, interleaved, CUDA events;
  2. the per-epoch weight hand-over: OperandGather refresh from the trainer's bucket against
     load_state_dict(trainer.state_dict()) + _pack (host round trip), host clock around a device synchronise;
  3. fit_head with 8 training and 4 validation tomograms, all resident: epoch wall clock with and without validation,
     epochs 1.. (epoch 0 reads the files and captures the CUDA graphs).

    python tools/val_probe.py [--reps 10] [--epochs 4] [--out val_probe.txt]
"""
from __future__ import annotations

import argparse
import functools
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

C, D, h, w = 1536, 128, 32, 32


def card() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown (nvidia-smi failed)"


@functools.lru_cache(maxsize=None)
def synthetic(seed: int):
    g = torch.Generator().manual_seed(seed)
    feats = torch.randn(C, D, h, w, generator=g).half()
    r = torch.rand(D, 16 * h, 16 * w, generator=g)
    lab = torch.where(r < 0.1, -1, (torch.rand(D, 16 * h, 16 * w, generator=g) < 0.3).long()).to(torch.int8)
    return feats, lab


def per_tomogram(head, reps: int, log):
    from cryovit_b200 import ops

    feats, lab = synthetic(0)
    feats, lab = feats.cuda(), lab.cuda()

    def fused():
        return head.score_volume(feats, lab)

    def unfused():
        _, probs = head.segment_volume(feats, want_logits=False)
        return ops.seg_stats(probs.view(-1), lab.float().view(-1), 0.5)

    a, b = fused(), unfused()
    counts = [1, 3, 4, 5, 6, 7]
    log(f"  sums agree: counts exact {torch.equal(a[counts], b[counts])}, soft rel diff "
        f"{float(((a[[0, 2]] - b[[0, 2]]).abs() / b[[0, 2]].abs()).max()):.2e}")
    times = {"score_volume": [], "segment_volume + labels + seg_stats": []}
    for _ in range(reps):
        for name, fn in (("score_volume", fused), ("segment_volume + labels + seg_stats", unfused)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1))
    for name, t in times.items():
        log(f"  {name}: median {statistics.median(t):.3f} ms, min {min(t):.3f}, max {max(t):.3f} ({reps} reps)")
    fm, um = statistics.median(times["score_volume"]), statistics.median(times["segment_volume + labels + seg_stats"])
    log(f"  difference (unfused - fused): {um - fm:+.3f} ms per tomogram")


def hand_over(reps: int, log):
    from cryovit_b200.head import CryoVITHeadB200
    from cryovit_b200.train import CryoVITHeadTrainerB200

    tr = CryoVITHeadTrainerB200(C)
    head = CryoVITHeadB200(C).cuda().attach_bucket(*tr.parameter_bucket())
    other = CryoVITHeadB200(C).cuda()
    t_g, t_l = [], []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        head.refresh()
        torch.cuda.synchronize()
        t_g.append(1e3 * (time.perf_counter() - t0))
        t0 = time.perf_counter()
        other.load_state_dict(tr.state_dict())
        torch.cuda.synchronize()
        t_l.append(1e3 * (time.perf_counter() - t0))
    log(f"  gather refresh: median {statistics.median(t_g):.2f} ms (min {min(t_g):.2f}, max {max(t_g):.2f})")
    log(f"  load_state_dict(trainer.state_dict()) + _pack: median {statistics.median(t_l):.2f} ms "
        f"(min {min(t_l):.2f}, max {max(t_l):.2f})")


def fit_epochs(epochs: int, log):
    from cryovit_b200.host.datasets import TomoDataset
    from cryovit_b200.host.fit import fit_head
    from cryovit_b200.host.metrics import DiceLoss, DiceMetric, F1Metric
    from cryovit_b200.host.validate import Validator

    class Synthetic(TomoDataset):
        """Tomograms generated from their record's seed instead of read from a file (same shapes and dtypes)."""

        def _load_tomogram(self, record):
            feats, lab = synthetic(int(record["seed"]))
            return {"sample": record["sample"], "tomo_name": record["tomo_name"], "input": feats.numpy(), "label": lab.numpy()}

    recs = [{"sample": "S", "tomo_name": f"t{i}", "seed": 100 + i} for i in range(12)]
    train = Synthetic(recs[:8], "dino_features", "mito", "split_id", "/nonexistent", train=True)
    val = Synthetic(recs[8:], "dino_features", "mito", "split_id", "/nonexistent", train=False)
    results = {}
    for tag in ("off", "on", "off", "on"):
        secs, hist = [], []
        v = Validator(val, C, {"dice_loss": DiceLoss()}, {"dice_metric": DiceMetric(), "f1_metric": F1Metric()}) if tag == "on" else None
        t0 = time.perf_counter()
        fit_head(train, in_channels=C, max_epochs=epochs, swa_epoch_start=None, epoch_seconds=secs, validator=v, val_history=hist)
        total = time.perf_counter() - t0
        val_s = [r["seconds"] for r in hist]
        steady = [s + (val_s[i] if val_s else 0.0) for i, s in enumerate(secs)][1:]
        results.setdefault(tag, []).append(statistics.mean(steady))
        log(f"  validation {tag}: training part per epoch {[round(s, 3) for s in secs]} s, validation "
            f"{[round(s, 3) for s in val_s]} s, epochs 1..{epochs - 1} wall clock mean {statistics.mean(steady):.3f} s, run {total:.1f} s")
        torch.cuda.empty_cache()
    log(f"  mean over the two runs: epoch wall clock without validation {statistics.mean(results['off']):.3f} s, with "
        f"{statistics.mean(results['on']):.3f} s (8 training steps, 4 validation tomograms)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--epochs", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    from cryovit_b200.head import CryoVITHeadB200
    from cryovit_b200.host.models import default_state_dict

    torch.cuda.set_device(0)
    log(f"card: {card()}")
    log(f"features {C}x{D}x{h}x{w} fp16, labels {D}x{16 * h}x{16 * w} int8")
    head = CryoVITHeadB200(C).load_state_dict(default_state_dict(C, seed=0)).cuda()
    log("1. per tomogram (CUDA events, interleaved)")
    per_tomogram(head, args.reps, log)
    del head
    log("2. per-epoch weight hand-over (host clock around a device synchronise)")
    hand_over(args.reps, log)
    log("3. fit_head, 8 training + 4 validation tomograms, resident")
    fit_epochs(args.epochs, log)
    log(f"card (end): {card()}")
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
