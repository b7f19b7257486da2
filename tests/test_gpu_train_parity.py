"""One training step of the head, tap by tap, against a float64 autograd restatement of the same graph.

The step (``CryoVITHeadTrainerB200.forward_backward``) is about 200 launches: forward convolutions, flipped and
transposed input-gradient convolutions, four weight-gradient kernel families, GroupNorm and GELU backward fused into
each other, pixel unshuffles. ``test_gpu_train.py`` checks each piece alone and the whole step on a 6-plane 4x4 crop,
where most dilated depth taps read only padding and the wide layers run single-CTA kernels. Here the step runs on crops
whose shapes reach what training reaches (``CASES``), with the default dispatch asserted from the shapes, and every
weight gradient is compared one 3x3x3 tap (or one 1x2x2 sub-pixel) at a time.

Tolerances come from a yardstick, not from guesses: the same float64 graph run a second time with every tensor the
trainer stores in bf16 rounded to bf16 (``_reference(bf16=True)``). Its distance from float64 says how far bf16 storage
alone moves each piece, and the trainer may be at most ``K`` times that far (``_bound``). Controls show that a lost
flip or a wrong tap order on any axis would break that bound.

What bf16 storage alone does is large where the gradient has passed several GroupNorm backward passes: with the
clip exercised, it moves the projection's gradient by 12-14 % and SB1's taps by up to 10 % from float64, and the trainer
lands as far (its error over the yardstick's is 0.9-1.2 there, at most 1.9 anywhere). In those pieces no tolerance can
resolve a 5 % error. A lost flip or a swapped tap changes a tap by the difference between two taps of the gradient,
and that difference can be small too: at case A's plane, SB2's kw-adjacent taps differ by less than twice its 3.4 %
noise, so a kw flip or a swapped kw pair there stays within the bound (x0.4-0.8). The controls are therefore asserted in
case B, which runs the same kernel instantiations with less noise (every edit breaks its bound, the weakest x1.6), and
printed for case A. A depth flip of the two full-resolution 8-channel output convolutions stays within the noise in
both cases (their kd = 0 and kd = 2 taps are nearly equal) and is printed only.

Measured on one B200 (1000 W power limit), the float64 reference of one step (forward + backward) takes 2.2 s and
10.8 GB above what is already allocated for case A (1536, 40, 32, 32), 0.25 s / 1.8 GB for B and 0.05 s / 0.4 GB for C;
the bf16 yardstick costs about as much again. The whole file runs in about 12 s.
"""
import time

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda"
F64, BF16 = torch.float64, torch.bfloat16

# Trainer error of a piece <= K x its bf16-yardstick error, capped at CAP (a 5 % error in a tap fails), except where
# bf16 storage alone moves the piece by more than CAP / NOISE_K: there NOISE_K x the yardstick. Never below FLOOR.
# Measured on one B200, worst trainer error / yardstick error over all pieces: 1.18 (case A), 1.89 (B, the per-channel
# error of a 16-channel bias), 1.68 (C); 0.90-1.18 where the yardstick exceeds CAP / NOISE_K. Loss error / yardstick
# error 0.93 (A), 0.84 (B), 0.90 (C); the loss yardsticks were 1.9e-5, 4.2e-6, 9.0e-7.
K = 4.0
NOISE_K = 2.0
FLOOR = 5e-3
CAP = 5e-2
LOSS_FLOOR = 1e-6

# C, D, h, w of the feature crop, feature dtype, and the dispatch each case must take (asserted from the shapes):
#   A  the production plane: 32x32 features = 8 row tiles per plane, so SB1's forward and input gradient run as CTA pairs;
#      rows8 / wgrad_tc8 at W = 512; D > 32, so every depth tap of every dilated convolution has in-volume voxels
#   B  CTA pairs with a partial border tile (BW 16 > W 12), a non-square plane, ragged row tiles at W = 24 .. 192
#   C  fp32 features: the non-cfirst projection and its weight gradient; D <= 24, so SB1's outer depth taps read only padding
CASES = {
    "A": dict(C=1536, D=40, h=32, w=32, dtype=torch.float16, pair=True, cfirst=True),
    "B": dict(C=384, D=36, h=16, w=12, dtype=torch.float16, pair=True, cfirst=True),
    "C": dict(C=384, D=20, h=8, w=8, dtype=torch.float32, pair=False, cfirst=False),
}


def _conv3_tiles(H: int, W: int) -> tuple[int, int]:
    """(row tiles per depth plane, BW) of the wide 3x3x3 convolution (csrc/gemm.cu, conv3_rows): BW is the smallest power
    of two >= min(W, 128), at least 8, and BH = 128 / BW. An even tile count selects the CTA-pair kernel."""
    BW = 8
    while BW < W and BW < 128:
        BW *= 2
    BH = 128 // BW
    return -(-H // BH) * -(-W // BW), BW


def _dispatch(C: int, D: int, h: int, w: int, dtype) -> dict:
    """The kernel choices of the trainer's default configuration that the cases are built to reach, from the shapes."""
    from cryovit_b200 import ops
    from cryovit_b200.head import BLOCKS

    tiles, bw = _conv3_tiles(h, w)
    narrow = []  # (cin, cout) of the 16 / 32-channel convolutions, forward and input gradient
    for c1, c2, _, _, _ in BLOCKS:
        for cin, cout in ((c1, c2), (c2, c2)):
            if max(cin, cout) <= 32:
                narrow += [(cin, cout), (cout, cin)]
    return {
        "sb1_pair": tiles % 2 == 0,
        "sb1_tiles_per_plane": tiles,
        "sb1_bw": bw,
        "full_res_w_mult8": (16 * w) % 8 == 0,
        "rows_narrow": bool(narrow) and all(ops.rows_supported(ci, co) for ci, co in narrow),
        # CryoVITHeadTrainerB200.forward_backward: the projection reads the (C, vox) fp16 volume as it lies
        "cfirst": dtype == torch.float16 and (D * h * w) % 8 == 0 and C % 8 == 0 and C >= 64,
    }


def _inputs(case: str, seed: int = 11):
    """State dict, features and labels of a case: randomised GroupNorm affines, output_layer.2 scaled so that about 30 % of
    the logits fall outside the clip's +-5, labels in {0, 1} with ignored planes at both depth ends and scattered ignored
    voxels."""
    from cryovit_b200.head import BLOCKS
    from oracle import head as ohead

    c = CASES[case]
    C, D, h, w = c["C"], c["D"], c["h"], c["w"]
    sd = ohead.random_state_dict(C, seed=seed)
    g = torch.Generator().manual_seed(seed)
    for bi, (c1, _, _, _, _) in enumerate(BLOCKS):
        p = f"layers.{bi + 2}.layers.0."
        sd[p + "weight"] = 1.0 + 0.3 * (2 * torch.rand(c1, generator=g) - 1)
        sd[p + "bias"] = 0.5 * (2 * torch.rand(c1, generator=g) - 1)
    gd = torch.Generator(device=DEV).manual_seed(seed)
    feats = (torch.randn(C, D, h, w, generator=gd, device=DEV) * 0.5).to(c["dtype"])
    H, W = 16 * h, 16 * w
    labels = (torch.rand(D, H, W, generator=gd, device=DEV) < 0.35).float()
    labels[:2] = -1
    labels[-2:] = -1
    labels[torch.rand(D, H, W, generator=gd, device=DEV) < 0.05] = -1
    # with default initialisation the logits sit within ~1e-2 of the bias: scale the last weight so that the 70th
    # percentile of |logit - bias| lands on the clip
    sd_dev = {k: v.to(DEV) for k, v in sd.items()}
    logits = ohead.forward_volume(sd_dev, feats.float()[None])[0, 0]
    dev = (logits - sd["output_layer.2.bias"].item()).abs().flatten()
    q = torch.quantile(dev[::max(1, dev.numel() // (1 << 22))], 0.70).item()
    sd["output_layer.2.weight"] = sd["output_layer.2.weight"] * (5.0 / q)
    assert all(sd[k].abs().min() > 0 for k in sd if k.endswith("bias"))
    return sd, feats, labels


class _Store(torch.autograd.Function):
    """Rounds to bf16 in the forward pass (a tensor the trainer stores in bf16) and / or the backward pass (its gradient)."""

    @staticmethod
    def forward(ctx, x, fwd: bool, bwd: bool):
        ctx.bwd = bwd
        return x.to(BF16).to(x.dtype) if fwd else x.clone()

    @staticmethod
    def backward(ctx, g):
        return (g.to(BF16).to(g.dtype) if ctx.bwd else g), None, None


def _reference(sd: dict, feats: torch.Tensor, labels: torch.Tensor, cfirst: bool, bf16: bool):
    """float64 autograd of CryoVITHeadTrainerB200.forward_backward on the GPU: projection + GELU, four SynthesisBlocks,
    output_layer.0 + GELU, output_layer.2, clip(-5, 5), sigmoid, masked Dice. ``bf16``: the yardstick run, where every
    activation, activation gradient and weight operand the trainer keeps in bf16 is rounded to bf16 (the projection
    weight of the cfirst path to fp16, its features as given; biases and GroupNorm affines stay exact).
    Returns (loss, {key: gradient}, fraction of the logits outside +-5)."""
    from cryovit_b200.head import BLOCKS

    P = {k: v.to(DEV, F64).requires_grad_(True) for k, v in sd.items()}
    if bf16:
        st = lambda t: _Store.apply(t, True, True)  # noqa: E731
        grad_only = lambda t: _Store.apply(t, False, True)  # noqa: E731
        wt = lambda t, dt=BF16: t + (t.detach().to(dt).to(F64) - t.detach())  # noqa: E731  (rounded value, exact gradient)
    else:
        st = grad_only = wt = lambda t, *_: t  # noqa: E731
    x = feats.to(F64)[None]
    if bf16 and not cfirst:
        x = x.to(BF16).to(F64)
    x = st(F.gelu(st(F.conv3d(x, wt(P["layers.0.weight"], torch.float16 if cfirst else BF16), P["layers.0.bias"]))))
    for bi, (c1, c2, c3, d1, d2) in enumerate(BLOCKS):
        p = f"layers.{bi + 2}.layers."
        x = st(F.group_norm(x, max(8, c1 // 8), P[p + "0.weight"], P[p + "0.bias"], 1e-3))
        x = st(F.gelu(st(F.conv3d(x, wt(P[p + "1.weight"]), P[p + "1.bias"], padding="same", dilation=(d1, 1, 1)))))
        x = st(F.gelu(st(F.conv3d(x, wt(P[p + "3.weight"]), P[p + "3.bias"], padding="same", dilation=(d2, 1, 1)))))
        x = st(F.gelu(st(F.conv_transpose3d(x, wt(P[p + "5.weight"]), P[p + "5.bias"], stride=(1, 2, 2)))))
    x = st(F.gelu(st(F.conv3d(x, wt(P["output_layer.0.weight"]), P["output_layer.0.bias"], padding="same"))))
    logits = grad_only(F.conv3d(x, wt(P["output_layer.2.weight"]), P["output_layer.2.bias"], padding="same"))[0, 0]
    prob = torch.sigmoid(torch.clip(logits, -5, 5))
    m = (labels > -1).to(F64)
    lab = labels.to(F64).clamp_min(0) * m
    loss = 1 - 2 * (lab * prob).sum() / (lab.sum() + (prob * m).sum() + 1e-3)
    loss.backward()
    clipped = (logits.detach().abs() > 5).to(F64).mean().item()
    return loss.item(), {k: v.grad for k, v in P.items()}, clipped


def _pieces(g: torch.Tensor) -> dict:
    """The pieces a gradient is compared in: each tap of a 3x3x3 weight, each sub-pixel of a 1x2x2 transposed-convolution
    weight, else the whole tensor. Tap weights also as a whole with the mean over their taps removed ("centred"): where
    one component common to every tap dominates (the 8-channel full-resolution layers), a wrong tap order changes each
    tap by less than the rounding noise of that component, but it changes how the taps differ from each other."""
    s = tuple(g.shape[2:])
    if s == (3, 3, 3):
        p = {f"tap{kd}{kh}{kw}": g[:, :, kd, kh, kw] for kd in range(3) for kh in range(3) for kw in range(3)}
    elif s == (1, 2, 2):
        p = {f"sub{i}{j}": g[:, :, 0, i, j] for i in range(2) for j in range(2)}
    else:
        return {"whole": g}
    p["centred"] = g - g.mean(dim=(2, 3, 4), keepdim=True)
    return p


def _rel(got: torch.Tensor, ref: torch.Tensor) -> float:
    """Relative Frobenius error; a zero reference must be matched exactly."""
    n = ref.norm().item()
    d = (got.to(F64) - ref).norm().item()
    return d / n if n > 0 else (0.0 if d == 0 else float("inf"))


def _chan(got: torch.Tensor, ref: torch.Tensor) -> float:
    """The largest per-output-channel error against the norm of the whole tensor."""
    return ((got.to(F64) - ref).reshape(ref.shape[0], -1).norm(dim=1).max() / ref.norm()).item()


def _bound(y: float) -> float:
    return max(min(K * y, CAP), NOISE_K * y, FLOOR)


def _compare(got: dict, ref: dict, yard: dict) -> tuple[list, dict]:
    """Rows (key, piece, error, yardstick, bound) for every piece and, for whole tensors, their per-channel error; and the
    bound of every (key, piece)."""
    rows, bounds = [], {}
    for k in ref:
        pr, pg, py = _pieces(ref[k]), _pieces(got[k]), _pieces(yard[k])
        for name in pr:
            y = _rel(py[name], pr[name])
            bounds[(k, name)] = _bound(y)
            rows.append((k, name, _rel(pg[name], pr[name]), y, bounds[(k, name)]))
            if name == "whole" and ref[k].numel() > 1:
                y = _chan(py[name], pr[name])
                rows.append((k, "channel", _chan(pg[name], pr[name]), y, _bound(y)))
    return rows, bounds


def _print_table(rows: list) -> None:
    """One line per parameter: its worst piece (by error / bound) and the worst error / yardstick ratio of its pieces."""
    print(f"  {'parameter':32s} {'pieces':>6s} {'worst piece':>11s} {'error':>10s} {'yardstick':>10s} {'bound':>9s} {'max ratio':>9s}")
    for k in dict.fromkeys(r[0] for r in rows):
        mine = [r for r in rows if r[0] == k]
        w = max(mine, key=lambda r: r[2] / r[4])
        ratio = max(r[2] / r[3] if r[3] > 0 else (0.0 if r[2] == 0 else float("inf")) for r in mine)
        print(f"  {k:32s} {len(mine):6d} {w[1]:>11s} {w[2]:10.3e} {w[3]:10.3e} {w[4]:9.2e} {ratio:9.2f}")


def _controls(ref: dict, bounds: dict) -> list:
    """Plain tensor edits of the reference's own weight gradients that a kernel bug of the kind this file guards against
    would produce: a lost flip along kd, kh or kw, two adjacent taps swapped, the two off-diagonal sub-pixels of a
    transposed convolution swapped. Returns (key, edit, worst error / bound over the pieces) for each."""

    def swap_taps(r):
        r = r.clone()
        r[:, :, 1, 1, [1, 2]] = r[:, :, 1, 1, [2, 1]]
        return r

    edits3 = {"flip kd": lambda r: r.flip(2), "flip kh": lambda r: r.flip(3), "flip kw": lambda r: r.flip(4),
              "swap tap 111/112": swap_taps}
    out = []
    for k, r in ref.items():
        s = tuple(r.shape[2:])
        edits = edits3 if s == (3, 3, 3) else {"swap sub 01/10": lambda r: r.transpose(3, 4)} if s == (1, 2, 2) else {}
        for name, f in edits.items():
            pe, pr = _pieces(f(r)), _pieces(r)
            out.append((k, name, max(_rel(pe[n], pr[n]) / bounds[(k, n)] for n in pr)))
    return out


@pytest.mark.parametrize("case", list(CASES))
def test_training_step_gradients_match_float64_tap_by_tap(cuda_lib, case):
    from cryovit_b200.head import BLOCKS
    from cryovit_b200.train import CryoVITHeadTrainerB200

    t_case = time.perf_counter()
    c = CASES[case]
    C, D, h, w = c["C"], c["D"], c["h"], c["w"]
    disp = _dispatch(C, D, h, w, c["dtype"])
    print(f"\n[train-parity {case}] features {tuple((C, D, h, w))} {c['dtype']}, dispatch {disp}")
    assert disp["sb1_pair"] == c["pair"] and disp["cfirst"] == c["cfirst"], disp
    assert disp["full_res_w_mult8"] and disp["rows_narrow"], disp

    sd, feats, labels = _inputs(case)
    tr = CryoVITHeadTrainerB200(C, state_dict=sd)
    assert set(tr.keys) == set(sd)
    loss = float(tr.forward_backward(feats, labels))
    got = {k: tr.g[k].to(F64) for k in tr.keys}
    del tr
    torch.cuda.synchronize()
    torch.cuda.empty_cache()

    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    ref_loss, ref, clipped = _reference(sd, feats, labels, c["cfirst"], bf16=False)
    torch.cuda.synchronize()
    ref_s, ref_gb = time.perf_counter() - t0, (torch.cuda.max_memory_allocated() - base) / 2 ** 30
    yard_loss, yard, _ = _reference(sd, feats, labels, c["cfirst"], bf16=True)
    ref = {k: ref[k] for k in got}
    print(f"[train-parity {case}] float64 reference: {ref_s:.2f} s, peak {ref_gb:.2f} GB above the baseline; "
          f"{100 * clipped:.1f} % of the logits outside +-5")

    rows, bounds = _compare(got, ref, yard)
    _print_table(rows)
    loss_err, loss_yard = abs(loss - ref_loss), abs(yard_loss - ref_loss)
    print(f"  loss {loss:.7f} float64 {ref_loss:.7f} bf16 yardstick {yard_loss:.7f}: error {loss_err:.2e}, yardstick {loss_yard:.2e}")
    ratios = [r[2] / r[3] for r in rows if r[3] > 0]
    print(f"[train-parity {case}] worst error / yardstick {max(ratios):.2f}; worst error / bound {max(r[2] / r[4] for r in rows):.3f}; "
          f"loss error / yardstick {loss_err / max(loss_yard, 1e-30):.2f}")

    # Controls: asserted in case B, which runs every kernel instantiation case A runs on a plane whose bf16 noise is
    # small enough to resolve each edit; at case A's production plane some are within that noise (module docstring),
    # so there they are printed only. A depth flip of the dilation-1 output convolutions is printed only everywhere.
    controls = _controls(ref, bounds) if case in ("A", "B") else []
    unseen = [x for x in controls if x[0].startswith("output_layer.") and x[1] == "flip kd"]
    controls = [x for x in controls if x not in unseen]
    missed = [x for x in controls if not x[2] > 1.0]
    if controls:
        print(f"[train-parity {case}] controls: {len(controls) - len(missed)} of {len(controls)} edits break their bounds, "
              f"the weakest x{min(x[2] for x in controls):.2f}; within: "
              + ", ".join(f"{k} {e} x{v:.2f}" for k, e, v in missed + unseen))

    # the point of each case, then the comparison, then the controls
    assert 0.2 <= clipped <= 0.4, clipped
    conv_keys = [f"layers.{bi + 2}.layers.{li}.weight" for bi in range(len(BLOCKS)) for li in (1, 3)]
    if case == "A":  # every depth tap of every dilated convolution reads in-volume voxels
        for k in conv_keys:
            n = [ref[k][:, :, kd].norm().item() for kd in range(3)]
            assert min(n[0], n[2]) >= 0.1 * n[1], (k, n)
    if case == "C":  # SB1's outer depth taps read only the TMA zero fill: anything else is a read outside the volume
        for k in conv_keys[:2]:
            for kd in (0, 2):
                assert torch.count_nonzero(ref[k][:, :, kd]) == 0, (k, kd)
                assert torch.count_nonzero(got[k][:, :, kd]) == 0, (k, kd, got[k][:, :, kd].abs().max().item())
    assert loss_err <= max(K * loss_yard, LOSS_FLOOR), (loss, ref_loss, yard_loss)
    bad = [r for r in rows if not r[2] <= r[4]]
    assert not bad, bad[:8]
    if case == "B":
        assert not missed, missed
    print(f"[train-parity {case}] {time.perf_counter() - t_case:.1f} s")


def test_grad_scale_and_graph_replay(cuda_lib, monkeypatch):
    """Case B. grad_scale (the 1/world factor of data parallelism) is a power of two here, exact in every rounding: four
    times the gradients at 0.25 must equal those at 1 up to what the atomic order changes between two runs. And the
    replay of the captured CUDA graph must fill the same gradient bucket as an eager step.

    The atomic-order difference is taken as the largest relative difference of any parameter between two eager runs:
    a single parameter's own difference is one draw of its summation order and can be zero by chance."""
    from cryovit_b200.train import CryoVITHeadTrainerB200

    monkeypatch.setenv("CVIT_TRAIN_GRAPH", "1")
    c = CASES["B"]
    sd, feats, labels = _inputs("B")
    tr = CryoVITHeadTrainerB200(c["C"], state_dict=sd)

    def grads(scale=None):
        tr.flat_g.fill_(float("nan"))  # a gradient the step does not write stays NaN
        if scale is not None:
            tr.forward_backward(feats, labels, scale)
        else:
            tr._forward_backward_graphed(feats, labels, 1.0)
        return {k: tr.g[k].clone() for k in tr.keys}

    def rel(a, b):
        return ((a - b).norm() / b.norm()).item()

    g1, g1b, g4 = grads(1.0), grads(1.0), grads(0.25)
    for _ in range(3):  # two eager steps, then the capture (which replays once)
        grads()
    assert len(tr._graphs) == 1 and all("graph" in e for e in tr._graphs.values()), "the step was not captured"
    gg = grads()  # one more replay
    noise = max(rel(g1b[k], g1[k]) for k in tr.keys)
    scaled = {k: rel(4 * g4[k], g1[k]) for k in tr.keys}
    replay = {k: rel(gg[k], g1[k]) for k in tr.keys}
    print(f"\n[train-parity] run-to-run {noise:.2e}; grad_scale 0.25 x 4 worst {max(scaled.values()):.2e}; "
          f"graph replay worst {max(replay.values()):.2e}")
    allowed = 2 * noise + 1e-7
    assert all(v <= allowed for v in scaled.values()), {k: v for k, v in scaled.items() if not v <= allowed}
    assert all(v <= allowed for v in replay.values()), {k: v for k, v in replay.items() if not v <= allowed}
