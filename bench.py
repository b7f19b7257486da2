#!/usr/bin/env python
"""Benchmark of the CryoVIT feature-extraction hot path on B200 (contract: see the task's bench.py section).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one synthetic tomogram: 128 slices of 512x512 uint8 -> DINOv2
ViT-g/14-reg4 features, fp16 (1536, 128, 32, 32) (BASELINE.json configs[1]; slice batch 128 as in the reference's
DinoFeaturesConfig.batch_size). Under torchrun each rank owns its own tomograms (BASELINE configs[2]: slices /
tomograms shard across GPUs with no data-path collective), so scaling is weak.

Numbers on the JSON line:
  value      slices/s with the raw tomogram already resident in HBM (CUDA events, max over ranks)
  e2e        slices/s through the public API extract_tomogram(np.uint8 host array) -> np.float16 host array,
             pinned H2D of the tomogram and D2H of the features inside the timed region
  roofline   the kernel with the largest share of the step, timed live with CUDA events inside the timed steps
  cpu_baseline  the fp32 oracle (a port: the reference cannot be imported here) on the box's host cores, bounded
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

MODEL = "dinov2_vitg14_reg"
D, H, W, BATCH = 128, 512, 512, 128
T, NP, C, FH, HEADS, DEPTH = 1029, 1024, 1536, 4096, 24, 40
# algorithmic work (BASELINE.md section 3)
FLOP_PER_SLICE = DEPTH * T * (2 * C * 3 * C + 2 * C * C + 2 * C * 2 * FH + 2 * FH * C + 4 * T * C) + 2 * 588 * C * NP
METRIC = "DINOv2 ViT-g/14 feature slices/sec"
# arithmetic type of the path per --operands mode (all accumulate in fp32 on the tensor cores, fp32 residual stream)
DTYPES = {"mixed-attn": "fp16 (norm1 out, attention out, qkv/proj weights) + bf16 (q/k/v, probabilities, norm2 out, w12, FFN hidden, w3) operands, fp32 accumulate",
          "mixed": "fp16 (LayerNorm out, attention out, qkv/proj/w12 weights) + bf16 (q/k/v, probabilities, FFN hidden, w3) operands, fp32 accumulate",
          "fp16": "fp16 (LayerNorm out, q/k/v, probabilities, attention out, qkv/proj/w12 weights) + bf16 (FFN hidden, w3) operands, fp32 accumulate",
          "bf16": "bf16 operands, fp32 accumulate"}


DUMP_POSITIONS = 4096  # --dump-outputs keeps 4096 of the 131072 feature vectors: 4096 x 1536 float32 = 25 MB


def dump_features(torch, feats, out_dir: str) -> None:
    """--dump-outputs: the (C, D, 32, 32) features of the last timed step, as whole C-channel feature vectors at a fixed
    seeded sample of (slice, row, column) positions, in flat position order: DIR/features_sample.npy, float32 (C, n).
    Two builds run with the same arguments see the same inputs, so their files compare element for element."""
    import numpy as np

    n = feats.shape[1] * feats.shape[2] * feats.shape[3]
    pos = np.sort(np.random.default_rng(0).choice(n, size=min(DUMP_POSITIONS, n), replace=False))
    sample = feats.reshape(feats.shape[0], n)[:, torch.from_numpy(pos).to(feats.device)]
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "features_sample.npy", sample.float().cpu().numpy())


def measured_peaks() -> tuple[dict, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text()), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region (recipe: B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# the workload both arms are quoted on (BASELINE config 2)
WORKLOAD = (f"ViT-g/14-reg4 (random init, LayerScale 1.0) features of one {D}x{H}x{W} uint8 tomogram per GPU per step, "
            f"slice batch {BATCH}, output fp16 ({C},{D},32,32)")



def config_dict(world: int) -> dict:
    """The SAME config object on both arms (the driver compares them key for key)."""
    return {"workload": WORKLOAD,
            "l2": "activations per step (>10 GB) exceed the 126 MB L2; no explicit flush needed",
            "parallelism": f"{world} independent replicas, tomograms sharded by rank, no collective"}


# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of the same
# kernels at the same shapes (profiles/r02_ncu_full_v1_*_kernels.json); bench.py itself never runs under ncu.
NCU_KEYS = {"linear_bias": "qkv_gemm", "attention": "attention", "linear_swiglu": "w12_swiglu", "layernorm": "layernorm",
            "proj_scale_residual": "proj_gemm", "w3_scale_residual": "w3_gemm"}


NCU_TRAFFIC_FILE = "r02_ncu_traffic.json"  # curated from profiles/r02_ncu_full_v3_*_kernels.json by tools/ncu_traffic_table.py


def ncu_traffic(kernel: str) -> float | None:
    p = ROOT / "profiles" / NCU_TRAFFIC_FILE
    if not p.exists() or kernel not in NCU_KEYS:
        return None
    for d in json.loads(p.read_text()):
        if d["kernel"] == NCU_KEYS[kernel]:
            return d["dram_bytes"]
    return None


class CallProfiler:
    """CUDA-event timing of EVERY call across the C ABI (``_lib.call``) while active: one record per launch with the
    symbol, its integer arguments (the shapes) and the events. Used for the per-layer tables of the head and of the
    training step (the ViT blocks have their own, lighter KernelTimer inside the timed region)."""

    # symbol -> (label, flops(int args)) ; int args are the call's integer arguments in order (pointers are skipped)
    @staticmethod
    def _conv(i):  # D, H, W, Cin, Cout(_pad), Cout_valid, dil -- ALGORITHMIC: all 27 taps, zero-padded ones included (SURVEY.md a13)
        return 2 * i[0] * i[1] * i[2] * 27 * i[3] * i[5]

    @staticmethod
    def executed_fraction(name: str, i) -> float:
        """Share of a dilated convolution's algorithmic FLOPs that the kernels execute: depth taps that fall outside
        [0, D) are skipped outright (with dilation 32 of 128 planes that is one tap in six)."""
        if "wgrad_mn" in name and i[6] == 27:  # K chunks whose depth tap leaves the volume are skipped
            D, dil = i[0], i[5]
        elif "conv3d_dilated" in name or "conv3d_halo" in name or "conv3d_wpackn" in name:
            D, dil = i[0], i[6]
        elif "conv3d_rows_ndhwc" in name:  # planes of a residue class outside the volume are skipped
            D, dil = i[0], i[5]
        else:
            return 1.0
        valid = sum((d - dil >= 0) + 1 + (d + dil < D) for d in range(D))
        return valid / (3.0 * D)

    FLOPS = {
        "cvit_linear_bias_cfirst_f16": lambda i: 2 * i[2] * i[3] * i[4],        # ldat, ldo, M, N, K, gelu
        "cvit_linear_bias_cfirst_f16_gn": lambda i: 2 * i[2] * i[3] * i[4],
        "cvit_linear_bias_gelu_bf16_gn": lambda i: 2 * i[2] * i[3] * i[4],
        "cvit_conv3d_dilated_ndhwc_tab": lambda i: CallProfiler._conv(i),
        "cvit_conv3d_halo_ndhwc_tab": lambda i: CallProfiler._conv(i),
        "cvit_conv3d_wpackn_ndhwc": lambda i: CallProfiler._conv(i),
        "cvit_convT_1x2x2_ndhwc_gn": lambda i: 2 * i[0] * i[1] * i[2] * i[3] * 4 * i[4],
        "cvit_linear_bias_fmt": lambda i: 2 * i[2] * i[3] * i[4],
        "cvit_linear_bias_bf16_nvalid": lambda i: 2 * i[2] * i[3] * i[4],
        "cvit_conv3d_dilated_ndhwc": lambda i: CallProfiler._conv(i),
        "cvit_conv3d_dilated_ndhwc_act": lambda i: CallProfiler._conv(i),
        "cvit_conv3d_halo_ndhwc": lambda i: CallProfiler._conv(i),
        "cvit_conv3d_halo_ndhwc_act": lambda i: CallProfiler._conv(i),
        "cvit_convT_1x2x2_ndhwc": lambda i: 2 * i[0] * i[1] * i[2] * i[3] * 4 * i[4],
        "cvit_convT_1x2x2_ndhwc_act": lambda i: 2 * i[0] * i[1] * i[2] * i[3] * 4 * i[4],
        "cvit_conv3d_wpack8_gelu": lambda i: 2 * i[0] * i[1] * i[2] * 27 * 64,
        "cvit_conv3d_wpack8_final": lambda i: 2 * i[0] * i[1] * i[2] * 27 * 8,
        "cvit_wgrad_splitk": lambda i: 2 * i[5] * i[0] * i[1] * i[2],           # M, N, k, lda, ldb, T
        "cvit_wgrad_narrow_ndhwc": lambda i: 2 * i[0] * i[1] * i[2] * 27 * i[3] * i[4],
        "cvit_wgrad_tc8_ndhwc": lambda i: 2 * i[0] * i[1] * i[2] * 27 * 64,                       # D, H, W, dil
        "cvit_wgrad_tcn_ndhwc": lambda i: 2 * i[0] * i[1] * i[2] * 27 * i[3] * i[4],              # D, H, W, Cin, Cout, dil
        "cvit_wgrad_mn_ndhwc": lambda i: 2 * i[0] * i[1] * i[2] * i[3] * i[4] * i[6],             # D, H, W, Ca, Cb, dil, ntaps, shift_a
        # the *_aux entry points (explicit activation mode + second tensor): same integer arguments, one more flag
        "cvit_linear_bias_cfirst_f16_aux": lambda i: 2 * i[2] * i[3] * i[4],
        "cvit_linear_bias_bf16_nvalid_aux": lambda i: 2 * i[2] * i[3] * i[4],
        "cvit_conv3d_dilated_ndhwc_aux": lambda i: CallProfiler._conv(i),
        "cvit_conv3d_halo_ndhwc_aux": lambda i: CallProfiler._conv(i),
        "cvit_conv3d_wpackn_ndhwc_aux": lambda i: CallProfiler._conv(i),
        "cvit_convT_1x2x2_ndhwc_aux": lambda i: 2 * i[0] * i[1] * i[2] * i[3] * 4 * i[4],
        "cvit_conv3d_wpack8_aux": lambda i: 2 * i[0] * i[1] * i[2] * 27 * 64,
        # one voxel per MMA row (csrc/conv_rows8.cu, csrc/conv_rows.cu)
        "cvit_conv3d_rows8": lambda i: 2 * i[0] * i[1] * i[2] * 27 * 64,                          # D, H, W, act
        "cvit_conv3d_rows8_final": lambda i: 2 * i[0] * i[1] * i[2] * 27 * 8,
        "cvit_conv3d_rows_ndhwc": lambda i: 2 * i[0] * i[1] * i[2] * 27 * i[3] * i[4],            # D, H, W, Cin, Cout, dil, act
    }

    def __init__(self, torch):
        from cryovit_b200 import _lib

        self.torch, self._lib, self.records, self.active = torch, _lib, [], False
        self._orig = _lib.call

        def wrapped(name, *a):
            if not self.active:
                return self._orig(name, *a)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            r = self._orig(name, *a)
            e.record()
            ints = tuple(int(x) for x in a[:-1] if isinstance(x, int) and not isinstance(x, bool) and abs(x) < (1 << 40))
            self.records.append((name, ints, s, e))
            return r

        _lib.call = wrapped

    def close(self):
        self._lib.call = self._orig

    def table(self, passes: int) -> list[dict]:
        """Launches of the profiled passes merged by (symbol, shape) in first-seen order; ms = per pass."""
        rows: dict = {}
        for name, ints, s, e in self.records:
            # device pointers are huge ints and were dropped above (< 2^40 keeps sizes, strides, flags)
            key = (name, ints)
            r = rows.setdefault(key, {"kernel": name.replace("cvit_", ""), "dims": list(ints), "ms": 0.0, "launches": 0})
            r["ms"] += s.elapsed_time(e)
            r["launches"] += 1
        out = []
        for (name, ints), r in rows.items():
            r["ms"] = round(r["ms"] / passes, 4)
            r["launches"] = r["launches"] // passes
            f = self.FLOPS.get(name)
            if f is not None:
                try:
                    r["tflops"] = round(f(ints) * r["launches"] / r["ms"] / 1e9, 1) if r["ms"] > 0 else None
                    r["flop"] = f(ints) * r["launches"]
                    ex = self.executed_fraction(name, ints)
                    if ex < 1.0:  # the algorithmic figure counts zero-padded depth taps the kernel skips
                        r["tflops_executed"] = round(r["tflops"] * ex, 1)
                except IndexError:
                    pass
            out.append(r)
        return out


def _roofline_of(rows: list[dict], peaks: dict, peak_src: str, traffic_file: str, what: str) -> dict | None:
    """Roofline block of the slowest tensor-core kernel of a per-layer table."""
    cand = [r for r in rows if r.get("tflops")]
    if not cand:
        return None
    top = max(cand, key=lambda r: r["ms"])
    # these kernels are timed one by one (an event pair per launch inside a 5-25 ms pass), not inside a long power-capped
    # step: the burst figure is their ceiling (MEASURED_PEAKS.json: bf16_tflops), the sustained one is quoted beside it
    peak = peaks.get("bf16_tflops", peaks.get("bf16_tflops_sustained"))
    sustained = peaks.get("bf16_tflops_sustained", peak)
    traffic, src = None, None
    p = ROOT / "profiles" / traffic_file
    if p.exists():
        for d in json.loads(p.read_text()):
            if d.get("kernel") == top["kernel"] and d.get("dims") == top["dims"]:
                traffic, src = d.get("dram_bytes"), f"profiles/{traffic_file} ({d.get('build', '?')})"
    executed = top.get("tflops_executed", top["tflops"])
    return {"kernel": f"{top['kernel']} {top['dims']}", "what": what, "bound": "tensor", "achieved": top["tflops"], "peak": peak,
            "unit": "TFLOP/s", "frac": round(executed / peak, 4), "frac_algorithmic": round(top["tflops"] / peak, 4),
            "achieved_executed": executed, "frac_vs_sustained": round(executed / sustained, 4), "peak_sustained": sustained,
            "note": "achieved counts the algorithmic FLOPs (all 27 taps, SURVEY.md a13); achieved_executed and frac discount the "
                    "zero-padded depth taps the kernel skips",
            "avg_launch_ms": round(top["ms"] / max(top["launches"], 1), 4), "flop_per_launch": top["flop"] // max(top["launches"], 1),
            "share_of_pass": round(top["ms"] / sum(r["ms"] for r in rows), 4), "traffic": traffic, "traffic_source": src,
            "peak_source": f"{peak_src} (burst bf16: kernel timed alone)"}


def head_cpu_baseline(torch) -> dict:
    """The oracle head (fp32, all host threads) on a (1536, 32, 28, 28) feature volume -> (32, 448, 448) logits,
    scaled to voxels/s (SURVEY.md 8d: head-1536 on a bounded volume, extrapolated linearly and labelled)."""
    from oracle import head as ohead

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = ohead.random_state_dict(1536, seed=0)
    x = torch.randn(1, 1536, 32, 28, 28, generator=torch.Generator().manual_seed(3)) * 0.5
    t0 = time.perf_counter()
    out = ohead.forward_volume(sd, x)
    dt = time.perf_counter() - t0
    vox = out.numel()
    return {"value": round(vox / dt, 0), "unit": "voxels/s", "cores": cores, "kind": "port",
            "sample": f"oracle head on one (1536,32,28,28) volume -> (32,448,448) logits in {dt:.1f} s; the full (1536,128,32,32) "
                      "volume scales linearly in voxels"}


def head_voxels_per_s(torch, dist=None, world: int = 1, steps: int = 3) -> dict:
    """CryoVIT 3-D head on one 1536-channel 128x32x32 feature volume (BASELINE config 4) -> 128x512x512 probabilities."""
    from cryovit_b200.head import CryoVITHeadB200, state_dict_keys

    g = torch.Generator().manual_seed(7)
    shapes = {"layers.0.weight": (1024, 1536, 1, 1, 1), "layers.0.bias": (1024,)}
    blocks = [(1024, 192, 128), (128, 64, 32), (32, 32, 32), (32, 16, 8)]
    for bi, (c1, c2, c3) in enumerate(blocks):
        p = f"layers.{bi + 2}.layers."
        shapes.update({p + "0.weight": (c1,), p + "0.bias": (c1,), p + "1.weight": (c2, c1, 3, 3, 3), p + "1.bias": (c2,),
                       p + "3.weight": (c2, c2, 3, 3, 3), p + "3.bias": (c2,), p + "5.weight": (c2, c3, 1, 2, 2),
                       p + "5.bias": (c3,)})
    shapes.update({"output_layer.0.weight": (8, 8, 3, 3, 3), "output_layer.0.bias": (8,),
                   "output_layer.2.weight": (1, 8, 3, 3, 3), "output_layer.2.bias": (1,)})
    sd = {}
    for k in state_dict_keys():
        shp = shapes[k]
        fan_in = 1
        for d in shp[1:]:
            fan_in *= d
        sd[k] = (torch.ones(shp) if k.endswith("0.weight") and len(shp) == 1 else
                 torch.randn(shp, generator=g) * (fan_in ** -0.5 if len(shp) > 1 else 0.02))
    head = CryoVITHeadB200(1536).load_state_dict(sd).cuda()
    feats = (torch.randn(1536, D, 32, 32, generator=g) * 0.5).half().cuda()
    for _ in range(2):
        head.segment_volume(feats, want_logits=False)
    torch.cuda.synchronize()
    l0 = head.launches
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        head.segment_volume(feats, want_logits=False)
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / steps
    if world > 1:  # every rank segments its own volume (tomograms shard by rank, no collective): max over ranks
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    vox = D * H * W
    head_voxels_per_s.head = head  # reused by pipeline_line
    line = {"value": round(world * vox / ms * 1e3, 0), "unit": "voxels/s (all GPUs)", "ms_per_volume": round(ms, 3),
            "tflops_per_gpu": round(94864 * vox / ms / 1e9, 1), "launches_per_volume": (head.launches - l0) // steps,
            "workload": f"CryoVIT head, one fp16 (1536,{D},32,32) feature volume per GPU -> ({D},{H},{W}) probabilities, weights random"}
    if int(os.environ.get("RANK", "0")) == 0:
        # per-layer table: two more passes with an event pair around every launch (outside the timed region above)
        prof = CallProfiler(torch)
        prof.active = True
        for _ in range(2):
            head.segment_volume(feats, want_logits=False)
        torch.cuda.synchronize()
        prof.active = False
        prof.close()
        rows = prof.table(2)
        peaks, peak_src = measured_peaks()
        line["frac_of_tensor_peak"] = round(line["tflops_per_gpu"] / peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]), 4)
        line["layers"] = [{k: r[k] for k in ("kernel", "dims", "ms", "launches", "tflops", "tflops_executed") if k in r} for r in rows]
        line["roofline"] = _roofline_of(rows, peaks, peak_src, "r02_ncu_traffic.json", "dominant kernel of the head forward")
    return line


def pipeline_line(torch, dist, world: int, vit, head, tomo_np, runs: int = 2) -> dict:
    """Tomogram in, mask out (SURVEY.md 8f row f3, the reference's dino_features + infer_model pair without the feature
    file in between): host uint8 (128,512,512) tomogram -> ViT-g features (stay in HBM) -> head -> uint8 mask on the
    host, through the public ``cryovit_b200.pipeline.segment_tomogram``; wall clock around the blocking call."""
    from cryovit_b200.pipeline import segment_tomogram

    segment_tomogram(tomo_np, vit, head, BATCH)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(runs):
        mask = segment_tomogram(tomo_np, vit, head, BATCH)
    sec = (time.perf_counter() - t0) / runs
    assert mask.shape == tomo_np.shape and mask.dtype.name == "uint8"
    if world > 1:
        t = torch.tensor([sec], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = float(t.item())
    return {"value": round(world * tomo_np.shape[0] / sec, 2), "unit": "slices/s (all GPUs), tomogram -> mask, host to host",
            "ms_per_tomogram": round(1e3 * sec, 2), "h2d_bytes_per_tomogram": int(tomo_np.size),
            "d2h_bytes_per_tomogram": int(mask.size),
            "workload": f"uint8 ({D},{H},{W}) tomogram -> ViT-g/14 features in HBM -> CryoVIT head -> uint8 mask, one tomogram per GPU"}


def head_train_voxels_per_s(torch, dist, world: int, steps: int = 3) -> dict:
    """BASELINE config 5: data-parallel CryoVIT head training, one (1536,128,32,32) feature crop + (128,512,512) labels
    per GPU and step: forward, masked DiceLoss, backward, one flat-bucket NCCL all-reduce (world > 1), AdamW."""
    from cryovit_b200.train import CryoVITHeadTrainerB200

    rank = int(os.environ.get("RANK", "0"))
    g = torch.Generator().manual_seed(500 + rank)
    feats = (torch.randn(1536, D, 32, 32, generator=g) * 0.5).half().cuda()
    labels = (torch.rand(D, H, W, generator=g) < 0.1).float()
    labels[::5] = -1  # 20 % of the slices unlabelled
    labels = labels.cuda()
    tr = CryoVITHeadTrainerB200(1536)
    for _ in range(4):  # two eager steps, the step that captures forward + backward into a CUDA graph, one replay
        loss = tr.train_step(feats, labels)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    l0 = tr.launches
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        loss = tr.train_step(feats, labels)
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / steps
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    vox = world * D * H * W
    line = {"value": round(vox / ms * 1e3, 0), "unit": "labelled-volume voxels/s (all GPUs)", "ms_per_step": round(ms, 2),
            "loss": round(float(loss), 5), "launches_per_step": (tr.launches - l0) // steps,
            "gradient_bucket_bytes": tr.flat_g.numel() * 4, "allreduce": "nccl, one flat fp32 bucket" if world > 1 else "none (1 GPU)",
            "workload": f"CryoVIT head training step, fp16 (1536,{D},32,32) crop + ({D},{H},{W}) labels per GPU, AdamW lr 1e-4 wd 1e-3, DiceLoss"}
    if rank == 0:
        # per-kernel table from one EAGER forward + backward (the timed steps above replay a CUDA graph, which events
        # cannot look into); gradients only, no optimizer step, so the trained state is not touched
        prof = CallProfiler(torch)
        tr.forward_backward(feats, labels, 1.0 / world)  # eager warm-up outside the profile
        torch.cuda.synchronize()
        prof.active = True
        tr.forward_backward(feats, labels, 1.0 / world)
        torch.cuda.synchronize()
        prof.active = False
        prof.close()
        rows = prof.table(1)
        peaks, peak_src = measured_peaks()
        top = sorted(rows, key=lambda r: -r["ms"])
        line["eager_forward_backward_ms"] = round(sum(r["ms"] for r in rows), 2)
        line["kernels"] = [{k: r[k] for k in ("kernel", "dims", "ms", "launches", "tflops") if k in r} for r in top if r["ms"] >= 0.05]
        line["model_tflops_per_step"] = round(3 * 94864 * D * H * W / 1e12, 2)
        line["frac_of_tensor_peak"] = round(3 * 94864 * D * H * W / ms / 1e9 / peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]), 4)
        line["roofline"] = _roofline_of(rows, peaks, peak_src, "r02_ncu_traffic.json", "dominant tensor-core kernel of one training step")
    return line


def cpu_oracle_slices_per_s(n_slices: int, sd=None, threads: int | None = None):
    """fp32 oracle (pre-processing + ViT-g forward + layout/cast) on the host cores over n_slices slices:
    (slices/s, cores, seconds, fp16 features)."""
    import numpy as np
    import torch

    from cryovit_b200.vit import CONFIGS, random_state_dict
    from oracle import dinov2 as odino
    from oracle import extract as oextract
    from oracle import preproc as opre

    cores = threads or os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = CONFIGS[MODEL]
    if sd is None:
        sd = random_state_dict(cfg, seed=0)
    tomo = np.random.default_rng(1234).integers(0, 256, size=(n_slices, H, W), dtype=np.uint8)
    model = odino.OracleDino(sd, cfg.num_heads)
    t0 = time.perf_counter()
    feats = oextract.dino_features(opre.dino_transform(opre.load_tomogram(tomo)), model, BATCH)
    dt = time.perf_counter() - t0
    assert feats.shape == (C, n_slices, 32, 32)
    return n_slices / dt, cores, dt, feats


def gpu_eager_baseline(torch, sd_cpu) -> dict:
    """The reference's own PyTorch path on THIS B200 (BASELINE.md section 4, SURVEY.md 2.2: "the number our kernels must
    beat"): the oracle modules moved to the GPU and run through stock torch / cuBLAS / cuDNN --
      * ViT-g: fp32 weights with TF32 matmuls (run/dino_features.py:24 set_float32_matmul_precision("high")), and again
        under bf16 autocast; attention through torch SDPA in both (the reference calls xformers
        memory_efficient_attention, which is not installed: SDPA is the same fused-attention class of kernel);
      * head: fp16 autocast (Lightning "16-mixed", config.py:70) over channels_last_3d tensors, cuDNN convolutions.
    Inputs are device resident (pre-processed slices / feature volume), i.e. these are kernel-only numbers to hold against
    ``value`` / ``head.value``, not against ``e2e``. None of our kernels run here."""
    import torch.nn.functional as F

    from cryovit_b200.vit import CONFIGS
    from oracle import dinov2 as odino
    from oracle import head as ohead

    cfg = CONFIGS[MODEL]
    out: dict = {"note": "oracle modules on the same GPU through stock torch (cuBLAS / cuDNN / SDPA); device-resident inputs"}
    orig_attn = odino._attention

    def sdpa_attention(x, sd, p, heads):  # upstream MemEffAttention: the fused kernel instead of the materialised softmax
        B, N, C = x.shape
        qkv = F.linear(x, sd[p + "attn.qkv.weight"], sd[p + "attn.qkv.bias"]).reshape(B, N, 3, heads, C // heads)
        q, k, v = qkv.permute(2, 0, 3, 1, 4)
        o = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(B, N, C)
        return F.linear(o, sd[p + "attn.proj.weight"], sd[p + "attn.proj.bias"])

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            fn()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / reps

    prec = torch.get_float32_matmul_precision()
    try:
        odino._attention = sdpa_attention
        sd = {k: v.cuda() for k, v in sd_cpu.items()}
        nb = 32
        x = torch.rand(nb, 3, 448, 448, device="cuda")
        torch.set_float32_matmul_precision("high")
        torch.backends.cudnn.allow_tf32 = True
        ms = timed(lambda: odino.forward_features(sd, x, cfg.num_heads), 2)
        out["vit_tf32"] = {"value": round(nb / ms * 1e3, 2), "unit": "slices/s", "ms_per_128_slices": round(ms * 128 / nb, 1),
                           "tflops": round(nb * FLOP_PER_SLICE / ms / 1e9, 1), "batch": nb,
                           "how": "fp32 weights, torch.set_float32_matmul_precision('high') as the reference, SDPA attention"}
        sd16 = {k: v.bfloat16() for k, v in sd.items()}
        del sd

        ms = timed(lambda: _bf16_vit(sd16, x, cfg.num_heads), 2)
        out["vit_bf16_autocast"] = {"value": round(nb / ms * 1e3, 2), "unit": "slices/s", "ms_per_128_slices": round(ms * 128 / nb, 1),
                                    "tflops": round(nb * FLOP_PER_SLICE / ms / 1e9, 1), "batch": nb,
                                    "how": "bf16 weights and activations (what torch.autocast(bfloat16) computes in), fp32 LayerNorm, SDPA"}
        del sd16, x
        torch.cuda.empty_cache()
    except Exception as err:  # noqa: BLE001 - a baseline that cannot run is reported, not fatal
        out["vit_error"] = f"{type(err).__name__}: {err}"[:300]
    finally:
        odino._attention = orig_attn
        torch.set_float32_matmul_precision(prec)
    try:
        hsd = {k: v.cuda() for k, v in ohead.random_state_dict(1536, seed=0).items()}
        feats = (torch.randn(1, 1536, D, 32, 32, device="cuda") * 0.5).to(memory_format=torch.channels_last_3d)

        def head_forward():
            with torch.autocast("cuda", dtype=torch.float16):
                return torch.sigmoid(_autocast_head(hsd, feats))

        ms = timed(head_forward, 2)
        out["head_fp16_autocast"] = {"value": round(D * H * W / ms * 1e3, 0), "unit": "voxels/s", "ms_per_volume": round(ms, 2),
                                     "tflops": round(94864 * D * H * W / ms / 1e9, 1),
                                     "how": "fp16 autocast (Lightning 16-mixed), channels_last_3d, cuDNN convolutions, fp32 GroupNorm"}
    except Exception as err:  # noqa: BLE001
        out["head_error"] = f"{type(err).__name__}: {err}"[:300]
    torch.cuda.empty_cache()
    return out


def _bf16_vit(sd16, x, heads):
    """oracle.dinov2.forward_features without its ``.float()`` of the weights: the same graph on bf16 tensors."""
    import torch
    import torch.nn.functional as F

    from oracle import dinov2 as odino

    with torch.no_grad():
        B = x.shape[0]
        C = sd16["cls_token"].shape[-1]
        t = F.conv2d(x.bfloat16(), sd16["patch_embed.proj.weight"], sd16["patch_embed.proj.bias"], stride=14)
        gh, gw = t.shape[-2:]
        t = t.flatten(2).transpose(1, 2)
        t = torch.cat([sd16["cls_token"].expand(B, -1, -1), t], dim=1)
        t = t + odino.interpolate_pos_encoding(sd16["pos_embed"], gh, gw).to(t.dtype)
        t = torch.cat([t[:, :1], sd16["register_tokens"].expand(B, -1, -1), t[:, 1:]], dim=1)
        depth = 1 + max(int(k.split(".")[1]) for k in sd16 if k.startswith("blocks."))
        for i in range(depth):
            p = f"blocks.{i}."
            t = t + sd16[p + "ls1.gamma"] * odino._attention(F.layer_norm(t, (C,), sd16[p + "norm1.weight"], sd16[p + "norm1.bias"], 1e-6), sd16, p, heads)
            t = t + sd16[p + "ls2.gamma"] * odino._ffn(F.layer_norm(t, (C,), sd16[p + "norm2.weight"], sd16[p + "norm2.bias"], 1e-6), sd16, p)
        return F.layer_norm(t, (C,), sd16["norm.weight"], sd16["norm.bias"], 1e-6)[:, 5:]


def _autocast_head(sd, x):
    """oracle.head.forward_volume without its ``.float()`` casts, so that autocast chooses the arithmetic."""
    import torch
    import torch.nn.functional as F

    from oracle.head import BLOCKS

    with torch.no_grad():
        x = F.gelu(F.conv3d(x, sd["layers.0.weight"], sd["layers.0.bias"]))
        for bi, (c1, c2, c3, d1, d2) in enumerate(BLOCKS):
            p = f"layers.{bi + 2}.layers."
            x = F.group_norm(x, max(8, c1 // 8), sd[p + "0.weight"], sd[p + "0.bias"], eps=1e-3)
            x = F.gelu(F.conv3d(x, sd[p + "1.weight"], sd[p + "1.bias"], padding="same", dilation=(d1, 1, 1)))
            x = F.gelu(F.conv3d(x, sd[p + "3.weight"], sd[p + "3.bias"], padding="same", dilation=(d2, 1, 1)))
            x = F.gelu(F.conv_transpose3d(x, sd[p + "5.weight"], sd[p + "5.bias"], stride=(1, 2, 2)))
        x = F.gelu(F.conv3d(x, sd["output_layer.0.weight"], sd["output_layer.0.bias"], padding="same"))
        x = F.conv3d(x, sd["output_layer.2.weight"], sd["output_layer.2.bias"], padding="same")
        return torch.clip(x, -5.0, 5.0)


def fit_loop_line(torch, dist, world: int, n_per_rank: int = 4, epochs: int = 3) -> dict:
    """The head's fit loop (host/fit.py: the schedule of configs/trainer/fit.yaml around the native training step) on
    tomogram FILES of BASELINE config 5's size: every rank owns ``n_per_rank`` files with fp16 (1536,128,32,32) features
    and int8 labels. Seconds per epoch with the training set resident in HBM after its first read (the default) against
    re-reading every file in every epoch (``cache_gb=0``: what the reference's loader does, tomo_dataset.py:89-146)."""
    import shutil
    import tempfile

    from cryovit_b200.host import fit, hdf
    from cryovit_b200.host.datasets import TomoDataset

    rank = int(os.environ.get("RANK", "0"))
    root = Path(tempfile.mkdtemp(prefix=f"cryovit_fit_r{rank}_"))
    try:
        g = torch.Generator(device="cuda").manual_seed(900 + rank)
        recs = []
        for i in range(n_per_rank):
            feats = (torch.randn(1536, D, 32, 32, device="cuda", generator=g) * 0.5).half().cpu().numpy()
            lab = (torch.rand(D, H, W, device="cuda", generator=g) < 0.3).to(torch.int8).cpu().numpy()
            hdf.write_tomogram(root / "S" / f"t{rank}_{i}.hdf", {"labels/mito": lab, "dino_features": feats})
            recs.append({"sample": "S", "tomo_name": f"t{rank}_{i}.hdf"})
        ds = TomoDataset(recs, "dino_features", "mito", "split_id", root, train=True)
        env_rank, env_world = os.environ.get("RANK"), os.environ.get("WORLD_SIZE")
        out = {}
        for label, gb in (("resident_in_hbm", None), ("files_every_epoch", 0.0)):
            secs: list = []
            # every rank trains on its own private files (same count): the rank sharding inside fit_head is switched off,
            # the gradient all-reduce is not (it looks at the process group, not at the environment)
            os.environ["RANK"], os.environ["WORLD_SIZE"] = "0", "1"
            try:
                fit.fit_head(ds, in_channels=1536, max_epochs=epochs, swa_epoch_start=None, cache_gb=gb, epoch_seconds=secs)
            finally:
                for k, v in (("RANK", env_rank), ("WORLD_SIZE", env_world)):
                    if v is None:
                        os.environ.pop(k, None)
                    else:
                        os.environ[k] = v
            t = torch.tensor(secs, device="cuda", dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            secs = t.tolist()
            out[label] = {"first_epoch_s": round(secs[0], 3), "later_epochs_s": [round(s, 3) for s in secs[1:]],
                          "ms_per_step_steady": round(min(secs[1:]) / n_per_rank * 1e3, 2)}
        out["workload"] = (f"{epochs} epochs over {n_per_rank} tomogram files per GPU (fp16 (1536,{D},32,32) features + int8 labels, "
                           f"{hdf.backend()} files on /tmp), one full-size crop per step, same crops and losses in both modes")
        out["speedup_steady"] = round(out["files_every_epoch"]["ms_per_step_steady"] / out["resident_in_hbm"]["ms_per_step_steady"], 2)
        return out
    finally:
        shutil.rmtree(root, ignore_errors=True)


def dataset_line(torch, dist, world: int, model, n_per_rank: int = 6) -> dict:
    """BASELINE config 3 through the FILES: every rank owns ``n_per_rank`` synthetic 128x512x512 uint8 tomogram files of
    one sample directory on the box's local disk and runs them through ``host.dino_features._process_sample`` -- the
    loop behind ``python -m cryovit.training.dino_features`` (reader / writer threads around the extractor, gzip of
    ``data``, 403 MB feature write per tomogram). Wall clock around the whole sample, max over ranks."""
    import shutil
    import tempfile

    import numpy as np

    from cryovit_b200.host import dino_features as df
    from cryovit_b200.host import hdf
    from cryovit_b200.host.config import compose

    rank = int(os.environ.get("RANK", "0"))
    root = Path(tempfile.mkdtemp(prefix=f"cryovit_ds_r{rank}_"))
    try:
        rng = np.random.default_rng(77 + rank)
        sample = "Q18"
        t0 = time.perf_counter()
        for i in range(n_per_rank):
            hdf.write_tomogram(root / "dino_features" / sample / f"tomo_{rank}_{i}.hdf",
                               {"data": rng.integers(0, 256, (D, H, W), dtype=np.uint8)})
        t_gen = time.perf_counter() - t0
        cfg = compose("dino_features", [f"paths.data_dir={root}", f"paths.exp_dir={root}/exp", f"sample={sample}", f"batch_size={BATCH}"])
        env_rank, env_world = os.environ.get("RANK"), os.environ.get("WORLD_SIZE")
        os.environ["RANK"], os.environ["WORLD_SIZE"] = "0", "1"  # this rank's private directory: no further sharding inside
        try:
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            done = df._process_sample(root / "dino_features", root / "tomograms", root / "csv", model, sample, cfg["datamodule"], BATCH)
            sec = time.perf_counter() - t0
        finally:
            for k, v in (("RANK", env_rank), ("WORLD_SIZE", env_world)):
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        assert len(done) == n_per_rank
        out_bytes = sum(f.stat().st_size for f in (root / "tomograms" / sample).iterdir())
        back = hdf.list_keys(root / "tomograms" / sample / done[0])
        assert sorted(back) == ["data", "dino_features"], back
        if world > 1:
            t = torch.tensor([sec], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t.item())
        return {"value": round(world * n_per_rank * D / sec, 2), "unit": "slices/s (all GPUs), tomogram FILES in -> feature FILES out, wall clock",
                "tomograms_per_gpu": n_per_rank, "seconds": round(sec, 2), "hdf_backend": hdf.backend(),
                "bytes_written_per_gpu": int(out_bytes), "write_GBps_per_gpu": round(out_bytes / sec / 1e9, 2),
                "source_generation_s": round(t_gen, 1), "disk": str(root.parent),
                "workload": f"BASELINE config 3 per GPU: {n_per_rank} x ({D},{H},{W}) uint8 files -> gzip data + fp16 ({C},{D},32,32) "
                            "dino_features per result file, read / write threads around the GPU extractor"}
    finally:
        shutil.rmtree(root, ignore_errors=True)


def config1_phantom(np):
    """Synthetic 32 x 448 x 448 uint8 tomogram with something to segment: bright 32-pixel blocks (two patches wide, four
    slices deep) on a dark background plus uniform noise, and the block mask as the label volume."""
    rng = np.random.default_rng(1234)
    coarse = rng.random((8, 14, 14)) < 0.3
    mask = np.repeat(np.repeat(np.repeat(coarse, 4, axis=0), 32, axis=1), 32, axis=2)
    tomo = 64.0 + 112.0 * mask + rng.integers(-48, 49, size=mask.shape)
    return np.clip(tomo, 0, 255).astype(np.uint8), mask.astype(np.float32)


def config1_line(torch, fit_steps: int = 150, fit_lr: float = 3e-4) -> dict:
    """BASELINE config 1 -- the reference's own CPU-runnable case, run in full on both sides: ViT-S/14-reg4 features of
    one synthetic 32 x 448 x 448 uint8 tomogram + the CryoVIT head over them. GPU: host tomogram in, host probabilities
    out, through the public calls (``extract_tomogram`` + ``segment_volume``). CPU: the oracle port on all host cores.
    The ViT is random init. A random-init head predicts one class everywhere (its logits sit within ~1e-2 of the output
    bias), which would make the mask comparison vacuous, so the head is first fitted for ``fit_steps`` AdamW steps
    (the B200 training path) to the phantom's block mask; both sides then load the SAME fitted weights. The two results
    are compared with BASELINE's tolerances."""
    import numpy as np

    from cryovit_b200.extract import extract_tomogram
    from cryovit_b200.head import CryoVITHeadB200
    from cryovit_b200.train import CryoVITHeadTrainerB200
    from cryovit_b200.vit import CONFIGS, build_model, random_state_dict
    from oracle import dinov2 as odino
    from oracle import extract as oextract
    from oracle import head as ohead
    from oracle import preproc as opre

    cfg = CONFIGS["dinov2_vits14_reg"]
    sd = random_state_dict(cfg, seed=0)
    tomo, labels = config1_phantom(np)
    model = build_model(cfg.name, sd).cuda()
    feats_dev = torch.from_numpy(extract_tomogram(tomo, model, batch_size=32)).cuda()
    trainer = CryoVITHeadTrainerB200(384, lr=fit_lr, state_dict=ohead.random_state_dict(384, seed=0))
    labels_dev = torch.from_numpy(labels).cuda()
    losses = [float(trainer.train_step(feats_dev, labels_dev)) for _ in range(fit_steps)]
    hsd = {k: v.detach().float().cpu().clone() for k, v in trainer.state_dict().items()}
    del trainer, feats_dev, labels_dev
    torch.cuda.empty_cache()
    head = CryoVITHeadB200(384).load_state_dict(hsd).cuda()

    def gpu_once():
        feats = extract_tomogram(tomo, model, batch_size=32)
        logits, probs = head.segment_volume(torch.from_numpy(feats).cuda())
        return feats, probs.cpu(), logits.cpu()

    gpu_once()
    torch.cuda.synchronize()
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        feats, probs, logits = gpu_once()
        ts.append(time.perf_counter() - t0)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    t0 = time.perf_counter()
    ref_feats = oextract.dino_features(opre.dino_transform(opre.load_tomogram(tomo)), odino.OracleDino(sd, cfg.num_heads), 32)
    ref_logits = ohead.forward_volume(hsd, torch.from_numpy(ref_feats).float()[None])[0, 0]
    cpu_s = time.perf_counter() - t0
    g, r = torch.from_numpy(feats.astype(np.float32)), torch.from_numpy(ref_feats.astype(np.float32))
    rel = ((g - r).norm(dim=0) / r.norm(dim=0)).max().item()
    cos = torch.nn.functional.cosine_similarity(g, r, dim=0).min().item()
    derr = (logits - ref_logits).abs()
    ref_mask, got_mask = torch.sigmoid(ref_logits) >= 0.5, probs >= 0.5
    agree = (got_mask == ref_mask).float().mean().item()
    lab = torch.from_numpy(labels) > 0.5
    gpu_s = sorted(ts)[1]
    return {"workload": "BASELINE config 1: ViT-S/14-reg4 features (random init) + CryoVIT head, one 32x448x448 uint8 phantom "
                        "tomogram, host buffers in and out; head fitted to the phantom's mask first, same weights on both sides",
            "gpu_ms": round(1e3 * gpu_s, 2), "cpu_s": round(cpu_s, 2), "cpu_cores": cores, "cpu_kind": "port",
            "feature_rel_err_max": round(rel, 5), "feature_cosine_min": round(cos, 6),
            "mask_agreement": round(agree, 5), "mask_positive_fraction": round(ref_mask.float().mean().item(), 4),
            "logit_abs_err_mean": round(derr.mean().item(), 5), "logit_abs_err_max": round(derr.max().item(), 5),
            "logit_std": round(ref_logits.std().item(), 4),
            "head_fit": {"steps": fit_steps, "lr": fit_lr, "dice_loss_first": round(losses[0], 4), "dice_loss_last": round(losses[-1], 4),
                         "mask_vs_labels_agreement": round((ref_mask == lab).float().mean().item(), 4)}}


def run_reference(args) -> None:
    """--impl reference: the reference's CPU path (oracle port) on the host cores; rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    sample = 2
    from cryovit_b200.vit import CONFIGS, random_state_dict

    sd = random_state_dict(CONFIGS[MODEL], seed=0)
    rates, cores = [], os.cpu_count()
    for i in range(args.warmup_ref + args.steps):
        r, cores, _, feats = cpu_oracle_slices_per_s(sample, sd)
        if i >= args.warmup_ref:
            rates.append(r)
    if args.dump_outputs:
        import torch

        dump_features(torch, torch.from_numpy(feats), args.dump_outputs)
    v = statistics.median(rates)
    line = {
        "impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": "slices/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup_ref, "ms_per_step": round(1e3 * sample / v, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args.gpus),
        "cpu_baseline": {"value": round(v, 4), "unit": "slices/s", "cores": cores, "kind": "port",
                         "sample": f"each step is a bounded sample of the workload: {sample} slices of {H}x{W} through preproc + "
                                   "ViT-g fp32 oracle + layout/cast, all host threads"},
        "e2e": {"value": round(v, 4), "unit": "slices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


class KernelTimer:
    """CUDA-event timing of the ops of ONE transformer block per step, inside the timed region."""

    def __init__(self, torch, ops_mod):
        self.torch, self.ops, self.records, self.active = torch, ops_mod, {}, False
        self._orig = {}

    FLOPS = {
        "linear_bias": lambda M: 2 * M * C * 3 * C,
        "attention": lambda M: 4 * (M // T) * HEADS * T * T * 64,
        "linear_swiglu": lambda M: 2 * M * C * 2 * FH,
    }

    def install(self):
        for name in ("layernorm", "linear_bias", "attention", "linear_scale_residual", "linear_swiglu"):
            orig = getattr(self.ops, name)
            self._orig[name] = orig

            def wrapped(*a, _orig=orig, _name=name, **k):
                if not self.active:
                    return _orig(*a, **k)
                key = _name
                if _name == "linear_scale_residual":
                    key = "proj_scale_residual" if a[0].shape[1] == C else "w3_scale_residual"
                s, e = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
                s.record()
                r = _orig(*a, **k)
                e.record()
                self.records.setdefault(key, []).append((s, e))
                return r

            setattr(self.ops, name, wrapped)

    def summary(self, M: int) -> dict:
        out = {}
        flops = {"linear_bias": 2 * M * C * 3 * C, "attention": 4 * (M // T) * HEADS * T * T * 64,
                 "linear_swiglu": 2 * M * C * 2 * FH, "proj_scale_residual": 2 * M * C * C,
                 "w3_scale_residual": 2 * M * FH * C}
        for k, evs in self.records.items():
            ms = statistics.mean(s.elapsed_time(e) for s, e in evs)
            out[k] = {"ms": ms, "flops": flops.get(k), "launches_timed": len(evs)}
        return out


def run_b200(args) -> None:
    import numpy as np
    import torch
    import torch.distributed as dist

    from cryovit_b200 import build, extract, ops
    from cryovit_b200.vit import CONFIGS, DinoVisionTransformerB200, random_state_dict

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL prints its version banner on the C-level stdout when the communicator is created; the contract is ONE
        # JSON line on stdout, so the banner is sent to stderr (fd-level redirect around init + first collective)
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    if rank == 0:
        build.build()
    if world > 1:
        dist.barrier()

    cfg = CONFIGS[MODEL]
    sd = random_state_dict(cfg, seed=0)
    model = DinoVisionTransformerB200(cfg, args.operands).load_state_dict(sd).cuda(local)
    if not (rank == 0 and world == 1 and not args.no_cpu_baseline):
        sd = None  # free 4.5 GB per rank unless the CPU baseline leg needs it
    g = torch.Generator().manual_seed(1234 + rank)
    tomo_host = torch.randint(0, 256, (D, H, W), generator=g, dtype=torch.uint8).pin_memory()
    tomo_dev = tomo_host.cuda(non_blocking=True)
    feats = torch.empty(C, D, 32, 32, device="cuda", dtype=torch.float16)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def step_device():
        extract.extract_tomogram_device(tomo_dev, model, BATCH, out=feats)

    # e2e goes through the public streaming API: host uint8 tomogram in, host fp16 features out, every step;
    # copies ride on their own streams under the previous / next tomogram's compute and ALL complete in the timed region
    stream = extract.TomogramFeatureStream(model, BATCH, depth=2)
    tomo_np = tomo_host.numpy()
    pending: list = []

    def step_e2e():
        pending.append(stream.submit(tomo_np))
        if len(pending) > 1:
            out = pending.pop(0).result()
            assert out.shape == (C, D, 32, 32)

    def drain_e2e():
        while pending:
            pending.pop(0).result()

    def timed(fn, steps, warmup, timer=None, drain=None):
        for _ in range(warmup):
            fn()
        if drain:
            drain()
        sync_all()
        launches0 = model.launches
        if timer:
            timer.active = True
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        t_wall0 = time.perf_counter()
        for _ in range(steps):
            fn()
        if drain:
            drain()  # every result is on the host before the clock stops
        e.record()
        torch.cuda.synchronize()
        wall_ms = (time.perf_counter() - t_wall0) * 1e3
        if timer:
            timer.active = False
        ms = s.elapsed_time(e)
        if drain:
            ms = max(ms, wall_ms)  # the copy streams' tail is covered by the host wait; take the longer clock
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        sync_all()
        return ms, model.launches - launches0

    # time only one block's kernels per step (block 20) so the event overhead stays negligible
    timer = KernelTimer(torch, ops)
    blocks = model._w["blocks"]
    timer.install()
    orig_blocks = model._blocks

    def blocks_with_probe(ws, B, T_):
        x = timer.active
        model._w["blocks"] = blocks[:20]
        timer.active = False
        orig_blocks(ws, B, T_)
        model._w["blocks"] = blocks[20:21]
        timer.active = x
        orig_blocks(ws, B, T_)
        timer.active = False
        model._w["blocks"] = blocks[21:]
        orig_blocks(ws, B, T_)
        model._w["blocks"] = blocks
        timer.active = x

    model._blocks = blocks_with_probe

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, launches = timed(step_device, args.steps, args.warmup, timer)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_features(torch, feats, args.dump_outputs)
    ms_e2e, _ = timed(step_e2e, args.steps, max(2, args.warmup // 2), drain=drain_e2e)

    # head inference and data-parallel head training: every rank takes part (training all-reduces its gradients)
    del stream
    torch.cuda.empty_cache()
    head_line = head_voxels_per_s(torch, dist, world)
    pipe_line = pipeline_line(torch, dist, world, model, head_voxels_per_s.head, tomo_np)
    del head_voxels_per_s.head
    torch.cuda.empty_cache()
    train_line = head_train_voxels_per_s(torch, dist, world)
    if not args.no_dataset:
        train_line["fit_loop"] = fit_loop_line(torch, dist, world)
    data_line = None if args.no_dataset else dataset_line(torch, dist, world, model)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    slices = world * D * args.steps
    value = slices / (ms / 1e3)
    e2e_value = slices / (ms_e2e / 1e3)
    peaks, peak_src = measured_peaks()
    ks = timer.summary(BATCH * T)
    per_step_ms = ms / args.steps
    shares = {k: v["ms"] * DEPTH / per_step_ms for k, v in ks.items()}
    # layernorm runs twice per block
    if "layernorm" in shares:
        shares["layernorm"] *= 1.0
    tensor_ks = {k: v for k, v in ks.items() if v["flops"]}
    top = max(tensor_ks, key=lambda k: tensor_ks[k]["ms"] * (1 if k != "layernorm" else 0)) if tensor_ks else None
    roof = None
    if top:
        tf = tensor_ks[top]["flops"] / tensor_ks[top]["ms"] / 1e9
        peak = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
        roof = {"kernel": top, "bound": "tensor", "achieved": round(tf, 1), "peak": peak, "unit": "TFLOP/s",
                "frac": round(tf / peak, 4), "peak_burst": peaks.get("bf16_tflops"),
                "frac_burst": round(tf / peaks["bf16_tflops"], 4) if peaks.get("bf16_tflops") else None,
                "traffic": ncu_traffic(top),
                "traffic_source": f"profiles/{NCU_TRAFFIC_FILE} (ncu --set full of the round's final library, capture r02 v3, one launch, "
                                  "same shapes)",
                "peak_source": f"{peak_src} (sustained bf16: kernel timed inside a long step)",
                "avg_launch_ms": round(tensor_ks[top]["ms"], 4)}
    kernels = {k: {"ms": round(v["ms"], 4), "tflops": round(v["flops"] / v["ms"] / 1e9, 1) if v["flops"] else None,
                   "share_of_step": round(shares[k] * (2 if k == "layernorm" else 1), 4)} for k, v in ks.items()}
    if "layernorm" in kernels and peaks.get("hbm_gbs"):
        # LayerNorm reads the fp32 residual stream once and writes the 16-bit operand: 6 bytes per element, nothing else
        ln_bytes = BATCH * T * C * 6
        gbps = ln_bytes / ks["layernorm"]["ms"] / 1e6
        kernels["layernorm"]["roofline"] = {"bound": "hbm", "achieved": round(gbps, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                            "frac": round(gbps / peaks["hbm_gbs"], 4), "algorithmic_bytes": ln_bytes,
                                            "traffic": ncu_traffic("layernorm")}
    for k in kernels:  # DRAM bytes per launch of every block kernel from the committed ncu capture
        if k != "layernorm" and ncu_traffic(k) is not None:
            kernels[k]["traffic"] = ncu_traffic(k)
    line = {
        "metric": METRIC, "value": round(value, 2), "unit": "slices/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(per_step_ms, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": DTYPES[args.operands], "data": "synthetic",
        "config": config_dict(world),
        "model_tflops": round(value * FLOP_PER_SLICE / 1e12, 1),
        "roofline": roof, "kernels": kernels, "clocks": clocks,
        "e2e": {"value": round(e2e_value, 2), "unit": "slices/s", "h2d_bytes_per_step": D * H * W,
                "d2h_bytes_per_step": C * D * 32 * 32 * 2},
        "gpu_launches": launches,
    }
    line["head"] = head_line
    line["pipeline"] = pipe_line
    line["head_train"] = train_line
    if data_line is not None:
        line["dataset"] = data_line
    del model
    torch.cuda.empty_cache()
    if world == 1 and not args.no_cpu_baseline:
        line["gpu_eager_baseline"] = gpu_eager_baseline(torch, sd)
        v, cores, dt, _ = cpu_oracle_slices_per_s(2, sd)
        line["cpu_baseline"] = {"value": round(v, 4), "unit": "slices/s", "cores": cores, "kind": "port",
                                "sample": f"2 slices of {H}x{W} through preproc + ViT-g fp32 oracle + layout/cast ({dt:.1f} s)"}
        del sd
        line["head"]["cpu_baseline"] = head_cpu_baseline(torch)
        line["config1"] = config1_line(torch)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU-oracle and GPU-eager baseline legs")
    ap.add_argument("--no-dataset", action="store_true", help="skip the file-based BASELINE config 3 leg")
    ap.add_argument("--operands", default="mixed-attn", choices=["mixed-attn", "mixed", "fp16", "bf16"],
                    help="16-bit formats of the ViT operands (cryovit_b200/vit.py): mixed-attn = fp16 norm1 / attention output and "
                         "the qkv / proj weights, everything else bf16 (default, the product path); mixed = the FFN input side fp16 too")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the features of the last one (a fixed "
                    "seeded sample of whole feature vectors) to DIR/features_sample.npy as float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    args.warmup_ref = min(args.warmup, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
