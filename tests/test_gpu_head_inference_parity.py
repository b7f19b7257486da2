"""Every launch of the inference forward (``CryoVITHeadB200.segment_volume``) against float64 of its own recorded operands.

The inference trunk runs machinery the trainer never runs (DESIGN §4.4, csrc/gn_fold.cu): GroupNorm statistics from the
producer's epilogue (``linear_bias_*_gn``, ``convT_1x2x2_gn``, the register-resident ``gn_direct`` sums of the 32-channel
transposed convolutions), ``gn_finalize`` -> scale / shift, ``gn_fold`` -> bf16 weights ``w * a_c`` in the consumer's layout
plus a 64-row bias table, and consumers that pick a table row per voxel from which of its taps fall inside the volume.
End-to-end checks (mean |dlogit| under 5 % of the logit std, 99.5 % mask agreement) absorb a table row that is wrong for
one border class or statistics that miss a block of rows. Here each launch is checked on its own recorded input, so
errors never compound:

* the ``ops`` entry points ``head.py`` calls are wrapped (monkeypatch): each wrapper clones its tensor arguments before
  the call and its outputs after it. The recorded sequence must be the default dispatch computed from the shapes, each
  launch's input must be bit-identical to the previous launch's output (a ping-pong aliasing bug fails here), and
  ``segment_volume``'s logits and probabilities must be the last launch's, bit for bit;
* every bf16 output obeys ``|got - ref| <= ulp_bf16(ref) + 1.13 * 2^-20 * S + 3e-5`` elementwise, with ``S`` the same
  float64 sum over ``|x| * |w|`` plus the absolute bias and shift terms (fp32 accumulation in any order), 1.13 the largest
  slope of GELU and 3e-5 the fitted-GELU error (``test_oracle.py::test_fast_gelu_formula``); the last two terms only
  where a GELU is applied. The mean signed error over the RMS of each output is bounded by ``MEAN_REL``;
* GroupNorm statistics: ``rstd = a / gamma`` and ``mean = (beta - b) / a`` from the kernel's scale / shift, against float64
  ``F.group_norm`` statistics (biased variance, eps 1e-3, consecutive channels, all four sub-pixels of a transposed
  convolution in their channel's group). The producer's epilogue sums its fp32 values BEFORE the bf16 store
  (gemm_tcgen05.cuh, ``gn_stats`` and ``gn_direct``), so the reference sums the float64 producer output, and the bound
  is the per-element bound above without the ulp term, plus fp32 accumulation of each partial sum ((n - 1) u of the
  sum of |terms|, n = 32 rows x cpg, or for ``gn_direct`` four times the values per thread the grid implies);
* ``gn_fold``: the bf16 weights must equal the image builder applied to ``w * a`` (fp32), bit for bit, and every one of
  the 64 table rows must match its float64 definition within 2^-20 of the sum of its absolute terms;
* convolutions after a fold: float64 conv of the RAW recorded input with the kernel's own folded weights, plus the bias,
  plus the shift computed independently of the table (a float64 conv of a volume equal to ``b_c`` inside and zero
  outside, with the fp32 weights);
* ``conv3d_rows8_final``: fp32 logits within the accumulation term, exactly +-5 wherever float64 lies beyond the clip
  (about 30 % of them), probabilities ``sigmoid(logit)`` within 1e-6.

Controls edit the float64 references the way each guarded bug would and require the edit to break its bound: for every
folded layer the interior table row used on the depth, the height and the width border in turn ("pad the raw tensor"),
depth dilation off by one and one dropped tap in every convolution, statistics that miss the first or the last (ragged)
32-row block or one sub-pixel column, and eps 1e-5 instead of 1e-3. Edits that change nothing in a case (dilation + 1
where no depth tap reaches the volume) are skipped; statistics edits that move a few parts in 10^5 of the production
volume's sums are asserted in the small cases and printed at production (``PRINT_ONLY``).

Cases (``CASES``): the production volume (every kernel at its production size: SB1 as CTA pairs, ``gn_direct`` at
128 x 256 x 256 x 32, rows8 at 512^2, D > 32 so every dilation sees all depth masks but "both depth taps out");
a shallow non-square fp32 volume (the ``features_to_ndhwc`` + ``linear_bias_gelu_gn`` projection, SB1 entirely in mask
dm = 0, SB2 with three depth classes, a single-CTA SB1 and ragged row tiles); one feature row (H = 1 at SB1: the
hm = 0 rows).

Measured on one B200 (1000 W power limit), seed 11:
* worst error / bound per launch kind, over the three cases: projection 0.510, conv3d_dilated_tab 0.507,
  conv3d_dilated 0.507, conv3d_rows after a fold 0.507, plain conv3d_rows 0.500, convT_1x2x2_gn 0.481, convT_1x2x2
  0.484, conv3d_rows8 0.451 (these sit at the ulp term: the outputs are correctly rounded bf16 of values within a
  fraction of the accumulation term), conv3d_rows8_final logits 0.062, probabilities 0.094, GroupNorm statistics 0.261
  (the projection's; 0.005-0.032 after a transposed convolution), fold tables 0.060. Mean signed error / RMS at most
  8.7e-5 (negative everywhere: the fitted GELU's bias). Folded weights bit-exact everywhere.
* controls, weakest margin per edit (production / shallow / one row): interior table row on the depth border x4940 /
  x5400 / x4530, height border x4940 / x5400 / x4530, width border x4150 / x4120 / x3120; dropped tap x128 / x93 / x126;
  depth dilation + 1 x256 / x268 / x255; sub-pixel column missed x106 / x87 / x71; eps 1e-5 x92 / x110 / x108;
  first 32-row block missed x0.58 (printed; x0.02-0.06 after the transposed convolutions) / x1.83 / x17; last (ragged)
  32-row block missed x0.58 (printed) / x1.89 / x17.
* the production case takes 3.0-5.6 s (about 2 s of float64 references, 17.3 GB at peak above the recorded
  launches), the whole file 11 s; 29.8-35.9 % of the logits lie beyond the clip.
"""
import inspect
import os
import time

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda"
F64, BF16 = torch.float64, torch.bfloat16

U = 2.0 ** -24     # fp32 unit roundoff
ACC = 2.0 ** -20   # fp32 accumulation in any order, relative to the sum of |terms|
G_ERR = 3e-5       # fitted GELU of every epilogue (DESIGN §4.4)
GELU_LIP = 1.13    # max |gelu'(x)| (1.129 at x = 2.42): an accumulation error leaves GELU at most this much larger
MEAN_REL = 3e-4    # |mean signed error| / RMS of the reference, per launch (measured at most 8.7e-5): a scale error of a
                   # few tenths of a percent of these positive-mean GELU outputs exceeds it
PROB_ABS = 1e-6    # probabilities against float64 sigmoid of the kernel's own logits (__expf + division)
EPS = 1e-3

CASES = {
    "production": dict(C=1536, D=128, h=32, w=32, dtype=torch.float16),
    "shallow": dict(C=384, D=20, h=6, w=5, dtype=torch.float32),
    "one_row": dict(C=1536, D=9, h=1, w=8, dtype=torch.float16),
}
# (case, control) pairs that are printed, not asserted: one 32-row block of the production volume is 1/4096 (projection)
# to 1/65536 (SB3's transposed convolution) of a group's values, below the GELU-fit term of the statistics bound
PRINT_ONLY = {("production", "stats: first 32-row block missed"), ("production", "stats: last 32-row block missed")}

TAPS = [(kd, kh, kw) for kd in range(3) for kh in range(3) for kw in range(3)]
OUTER_DEPTH = [t for t in TAPS if t[0] != 1]
DROPPED = (1, 1, 2)

WATCHED = ("linear_bias_cfirst_gn", "linear_bias_gelu_gn", "features_to_ndhwc", "groupnorm_fold", "conv3d_dilated_tab",
           "conv3d_dilated", "conv3d_rows", "convT_1x2x2_gn", "convT_1x2x2", "conv3d_rows8", "conv3d_rows8_final")
# entry points of the non-default arms: recorded too, so that a launch the dispatch does not expect is seen
OTHERS = ("linear_bias", "linear_bias_cfirst", "groupnorm_ndhwc", "conv3d_halo", "conv3d_halo_tab", "conv3d_wpackn",
          "conv3d_wpack8_gelu", "conv3d_wpack8_final", "head_out_conv")
OUTPUTS = {"groupnorm_fold": ("ab", "w_out", "table"), "linear_bias_cfirst_gn": ("out", "partials"),
           "linear_bias_gelu_gn": ("out", "partials"), "convT_1x2x2_gn": ("out", "partials"),
           "conv3d_rows8_final": ("logits", "probs")}


def _inputs(case: str, seed: int = 11):
    """State dict and features of a case (the recipe of test_gpu_train_parity._inputs): GroupNorm affines gamma in 1 +- 0.3
    and beta in +-0.5, so that the folded shift is far from zero; output_layer.2 scaled so that about 30 % of the logits
    fall outside the clip's +-5."""
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
    # with default initialisation the logits sit within ~1e-2 of the bias: scale the last weight so that the 70th
    # percentile of |logit - bias| lands on the clip
    sd_dev = {k: v.to(DEV) for k, v in sd.items()}
    logits = ohead.forward_volume(sd_dev, feats.float()[None])[0, 0]
    dev = (logits - sd["output_layer.2.bias"].item()).abs().flatten()
    q = torch.quantile(dev[::max(1, dev.numel() // (1 << 22))], 0.70).item()
    sd["output_layer.2.weight"] = sd["output_layer.2.weight"] * (5.0 / q)
    assert all(sd[k].abs().min() > 0 for k in sd if k.endswith("bias"))
    return sd, feats


def _expected_dispatch(C: int, D: int, h: int, w: int, dtype) -> list:
    """The launches of segment_volume's default configuration, from the shapes (as test_gpu_train_parity._dispatch)."""
    from cryovit_b200 import ops
    from cryovit_b200.head import BLOCKS

    cfirst = dtype == torch.float16 and (D * h * w) % 8 == 0 and C % 8 == 0 and C >= 64
    seq = ["linear_bias_cfirst_gn"] if cfirst else ["features_to_ndhwc", "linear_bias_gelu_gn"]
    for bi, (c1, c2, _, _, _) in enumerate(BLOCKS):
        if ops.rows_supported(c1, c2) and ops.rows_supported(c2, c2):  # 16 / 32 channels: one voxel per MMA row
            seq += [("groupnorm_fold", ops.LAYOUT_ROWS), "conv3d_rows", "conv3d_rows"]
        else:  # wide layers: the implicit-GEMM tap convolution
            seq += [("groupnorm_fold", ops.LAYOUT_TAPS), "conv3d_dilated_tab", "conv3d_dilated"]
        seq.append("convT_1x2x2_gn" if bi + 1 < len(BLOCKS) else "convT_1x2x2")
    assert (16 * w) % 8 == 0  # full-resolution planes on conv_rows8.cu
    return seq + ["conv3d_rows8", "conv3d_rows8_final"]


def _record(monkeypatch) -> list:
    """Wrap the head's ops entry points: (name, arguments cloned before the call, outputs cloned after it, return value)."""
    from cryovit_b200 import ops

    log = []

    def wrap(name, fn):
        sig = inspect.signature(fn)

        def rec(*args, **kwargs):
            ba = sig.bind(*args, **kwargs)
            ba.apply_defaults()
            inp = {k: v.clone() if isinstance(v, torch.Tensor) else v for k, v in ba.arguments.items()}
            ret = fn(*args, **kwargs)
            out = {k: ba.arguments[k].clone() for k in OUTPUTS.get(name, ("out",)) if isinstance(ba.arguments.get(k), torch.Tensor)}
            log.append((name, inp, out, ret))
            return ret

        return rec

    for name in WATCHED + OTHERS:
        monkeypatch.setattr(ops, name, wrap(name, getattr(ops, name)))
    return log


def _bits(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view({torch.bfloat16: torch.int16, torch.float16: torch.int16, torch.float32: torch.int32,
                                torch.float64: torch.int64}[t.dtype])


def _same(a: torch.Tensor, b: torch.Tensor) -> bool:
    return a.dtype == b.dtype and a.shape == b.shape and a.device == b.device and torch.equal(_bits(a), _bits(b))


def _ulp_bf16(x: torch.Tensor) -> torch.Tensor:
    """Spacing of bf16 numbers in the binade of x (8 significant bits); 0 at 0."""
    _, e = torch.frexp(x)
    return torch.where(x == 0, torch.zeros_like(x), torch.exp2((e - 8).to(F64)))


def _conv64(x: torch.Tensor, w: torch.Tensor, dil: int, taps=TAPS, shape=None) -> torch.Tensor:
    """float64 "same" 3x3x3 convolution with depth dilation ``dil``, channels last: x [D, H, W, Cin], w [Cout, Cin, 3, 3, 3]
    -> [D, H, W, Cout], the sum over ``taps`` of shifted(x) @ w_tap^T; the zero padding is done by slicing. With ``shape``,
    x is a [Cin] vector standing for a volume of that shape equal to x inside and zero outside."""
    D, H, W = shape if shape is not None else x.shape[:3]
    out = torch.zeros(D, H, W, w.shape[0], dtype=F64, device=w.device)
    for kd, kh, kw in taps:
        od, oh, ow = (kd - 1) * dil, kh - 1, kw - 1  # output (d, h, w) reads input (d + od, h + oh, w + ow)
        d0, d1, h0, h1, w0, w1 = max(0, -od), min(D, D - od), max(0, -oh), min(H, H - oh), max(0, -ow), min(W, W - ow)
        if d0 >= d1 or h0 >= h1 or w0 >= w1:
            continue
        wt = w[:, :, kd, kh, kw].t()
        src = x if shape is not None else x[d0 + od:d1 + od, h0 + oh:h1 + oh, w0 + ow:w1 + ow]
        out[d0:d1, h0:h1, w0:w1] += src @ wt
    return out


def _masks(n: int, dil: int) -> set:
    """Mask values (bit 0: the lower tap is inside, bit 1: the upper tap) that positions 0..n-1 of an axis take."""
    return {(1 if i >= dil else 0) | (2 if i + dil < n else 0) for i in range(n)}


def _rows_reached(D: int, H: int, W: int, dil: int) -> set:
    return {(dm * 4 + hm) * 4 + wm for dm in _masks(D, dil) for hm in _masks(H, 1) for wm in _masks(W, 1)}


def _taps_from_image(w_taps: torch.Tensor, cout: int, cin: int) -> torch.Tensor:
    """LAYOUT_TAPS weights [27 * cout_pad, cin] (tap = (kd*3 + kh)*3 + kw) -> [cout, cin, 3, 3, 3]."""
    return w_taps.reshape(27, -1, cin)[:, :cout].permute(1, 2, 0).reshape(cout, cin, 3, 3, 3)


class _Case:
    """Per-case tables: launch rows (label, kind, worst error / bound, mean signed error / RMS) and controls (label, edit,
    margin = worst |got - edited reference| / bound)."""

    def __init__(self, name):
        self.name, self.rows, self.controls = name, [], []

    def check(self, label, kind, got, pre, S, gelu: bool):
        """Elementwise bound of a bf16 output; returns (reference, bound) for the controls."""
        ref = F.gelu(pre) if gelu else pre
        bound = _ulp_bf16(ref) + (GELU_LIP if gelu else 1.0) * ACC * S + (G_ERR if gelu else 0.0)
        err = got.to(F64) - ref
        self.rows.append((label, kind, (err.abs() / bound).max().item(), (err.mean() / ref.square().mean().sqrt()).item()))
        return ref, bound

    def control(self, label, edit, got, ref_edit, bound):
        self.controls.append((label, edit, ((got.to(F64) - ref_edit).abs() / bound).max().item()))

    def conv_controls(self, label, got, x64, w64, pre, bound, dil, gelu=True, clip=False):
        """One dropped tap and (where a depth tap reaches the volume) depth dilation + 1, as edits of the pre-activation."""
        act = (lambda t: F.gelu(t)) if gelu else (lambda t: t.clamp(-5.0, 5.0)) if clip else (lambda t: t)
        self.control(label, f"tap {DROPPED} dropped", got, act(pre - _conv64(x64, w64, dil, taps=[DROPPED])), bound)
        if x64.shape[0] > dil:
            moved = pre - _conv64(x64, w64, dil, taps=OUTER_DEPTH) + _conv64(x64, w64, dil + 1, taps=OUTER_DEPTH)
            self.control(label, "depth dilation + 1", got, act(moved), bound)


def _linear64(a: torch.Tensor, w: torch.Tensor, b: torch.Tensor):
    """a [M, K], w [N, K], b [N] -> float64 a w^T + b and the same sum over absolute values."""
    a64, w64, b64 = a.to(F64), w.to(F64), b.to(F64)
    return a64 @ w64.t() + b64, a64.abs() @ w64.abs().t() + b64.abs()


def _check_stats(cs: _Case, label: str, prod: dict, fa: dict, ab: torch.Tensor, G: int, eps: float):
    """The fold's scale / shift against float64 group statistics of the producer's output, and the statistics controls.
    prod: y [rows, reps, C] float64 producer output (post-GELU, pre-rounding), B [same] bound on the kernel's fp32 value,
    n_acc: fp32 terms per partial sum."""
    y, B, n_acc = prod["y"], prod["B"], prod["n_acc"]
    rows, reps, C = y.shape
    cpg = C // G
    n = rows * reps * cpg
    assert fa["n_per_group"] == n, (fa["n_per_group"], n)

    def gs(t):  # [rows, reps, C] -> per-row group sums [rows, G]
        return t.reshape(rows, reps, G, cpg).sum(dim=(1, 3))

    s1r, s2r = gs(y), gs(y * y)
    s1, s2 = s1r.sum(0), s2r.sum(0)
    sum_b, sum_yb, sum_ya = gs(B).sum(0), gs(2 * y.abs() * B + B * B).sum(0), gs(y.abs()).sum(0)

    def stats(t1, t2, e=eps):
        mu = t1 / n
        return mu, 1.0 / (t2 / n - mu * mu + e).sqrt()

    mu, rstd = stats(s1, s2)
    var = s2 / n - mu * mu
    dmu = (sum_b + n_acc * U * sum_ya) / n
    dvar = (sum_yb + (n_acc + 1) * U * s2) / n + 2 * mu.abs() * dmu + dmu * dmu
    r = dvar / (var + eps)
    assert r.max().item() < 0.5, r.max().item()
    a, b = ab[:C].to(F64), ab[C:2 * C].to(F64)
    gamma, beta = fa["gamma"].to(F64), fa["beta"].to(F64)
    rstd_k, mu_k = (a / gamma).view(G, cpg), ((beta - b) / a).view(G, cpg)
    rstd_b = ((0.5 * r / (1 - r) + 4 * U) * rstd)[:, None]
    mu_b = dmu[:, None] + 4 * U * (mu.abs()[:, None] + (b / a).abs().view(G, cpg))

    def ratio(m, s):
        return max(((mu_k - m[:, None]).abs() / mu_b).max().item(), ((rstd_k - s[:, None]).abs() / rstd_b).max().item())

    cs.rows.append((label, "groupnorm stats", ratio(mu, rstd), float("nan")))
    last = (rows - 1) // 32 * 32
    edits = {"stats: first 32-row block missed": stats(s1 - s1r[:32].sum(0), s2 - s2r[:32].sum(0)),
             "stats: last 32-row block missed": stats(s1 - s1r[last:].sum(0), s2 - s2r[last:].sum(0)),
             "stats: eps 1e-5": stats(s1, s2, 1e-5)}
    if reps == 4:
        y3 = y[:, 3].reshape(rows, G, cpg)
        edits["stats: sub-pixel (1,1) missed"] = stats(s1 - y3.sum((0, 2)), s2 - y3.square().sum((0, 2)))
    for k, (m, s) in edits.items():
        cs.controls.append((label, k, ratio(m, s)))


def _check_fold(cs: _Case, label: str, fa: dict, fo: dict, w32: torch.Tensor, layout: int, coutp: int):
    """gn_fold: folded weights bit for bit, all 64 table rows against their float64 definition. w32: fp32 [cout, cin, 3, 3, 3]
    as loaded. Returns the kernel's shift b [cin] (float64)."""
    from cryovit_b200 import ops
    from cryovit_b200.head import _conv_taps, rowsn_weight_image

    cout, cin = w32.shape[:2]
    build = (lambda t: _conv_taps(t, coutp).reshape(-1)) if layout == ops.LAYOUT_TAPS else rowsn_weight_image
    assert _same(fa["w32"].cpu(), build(w32)), f"{label}: the fold's fp32 weight image is not the layer's weight"
    a = fo["ab"][:cin].cpu()
    assert _same(fo["w_out"].cpu(), build(w32 * a.view(1, cin, 1, 1, 1)).to(BF16)), f"{label}: folded weights differ from bf16(w * a)"
    bsh = fo["ab"][cin:2 * cin].to(F64)
    wp = torch.zeros(coutp, cin, 3, 3, 3, dtype=F64, device=DEV)
    wp[:cout] = w32.to(DEV, F64)
    per_tap = torch.einsum("oct,c->to", wp.reshape(coutp, cin, 27), bsh)  # [27, coutp]
    per_tap_abs = torch.einsum("oct,c->to", wp.reshape(coutp, cin, 27).abs(), bsh.abs())
    bias = fa["bias"].to(F64)
    ref, S = torch.empty(64, coutp, dtype=F64, device=DEV), torch.empty(64, coutp, dtype=F64, device=DEV)
    for m in range(64):
        inside = [((m >> 4) & 3, (m >> 2) & 3, m & 3)]
        sel = [(kd * 3 + kh) * 3 + kw for kd, kh, kw in TAPS
               if all(k == 1 or (k == 0 and msk & 1) or (k == 2 and msk & 2) for k, msk in zip((kd, kh, kw), inside[0]))]
        ref[m] = bias + per_tap[sel].sum(0)
        S[m] = bias.abs() + per_tap_abs[sel].sum(0)
    got = fo["table"].view(64, coutp).to(F64)
    cs.rows.append((label, "fold table", ((got - ref).abs() / (ACC * S)).max().item(), float("nan")))
    return bsh


@pytest.mark.parametrize("case", list(CASES))
def test_segment_volume_launches_match_float64(cuda_lib, case, monkeypatch):
    from cryovit_b200 import ops
    from cryovit_b200.head import BLOCKS, CryoVITHeadB200, rows8_weight_image, rowsn_weight_image

    t_case = time.perf_counter()
    c = CASES[case]
    C, D, h, w, dtype = c["C"], c["D"], c["h"], c["w"], c["dtype"]
    for k in list(os.environ):
        if k.startswith("CVIT_HEAD_"):
            monkeypatch.delenv(k)
    sd, feats = _inputs(case)
    log = _record(monkeypatch)
    head = CryoVITHeadB200(C).load_state_dict(sd).cuda()
    logits, probs = head.segment_volume(feats)
    torch.cuda.synchronize()
    del head
    torch.cuda.empty_cache()
    t_ref = time.perf_counter()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()

    # ------------------------------------------------------------------ dispatch
    seq = [(n, a["layout"]) if n == "groupnorm_fold" else n for n, a, _, _ in log]
    expected = _expected_dispatch(C, D, h, w, dtype)
    print(f"\n[head-inference {case}] features {(C, D, h, w)} {dtype}: {len(log)} launches recorded")
    assert seq == expected, (seq, expected)

    cs = _Case(case)
    it = iter(log)
    vox0 = D * h * w
    with torch.no_grad():
        # -------------------------------------------------------------- projection
        if seq[0] == "linear_bias_cfirst_gn":
            _, pa, po, _ = next(it)
            assert _same(pa["at"], feats.reshape(C, vox0))
            A = pa["at"].t()
        else:
            _, ta, to, _ = next(it)
            assert _same(ta["features"], feats)
            assert _same(to["out"], feats.permute(1, 2, 3, 0).to(BF16)), "features_to_ndhwc is a transpose and a rounding: exact"
            _, pa, po, _ = next(it)
            assert _same(pa["a"], to["out"].reshape(vox0, C))
            A = pa["a"]
        pre, S = _linear64(A, pa["w"], pa["bias"])
        ref, _ = cs.check("proj", "linear+gelu", po["out"].view(vox0, 1024), pre, S, gelu=True)
        cpg0 = pa["cpg"]
        prod = {"y": ref.view(vox0, 1, 1024), "B": (GELU_LIP * ACC * S + G_ERR).view(vox0, 1, 1024),
                "partials": po["partials"], "n_acc": 32 * cpg0}
        del pre, S, ref, A
        cur = po["out"].view(D, h, w, 1024)

        # -------------------------------------------------------------- synthesis blocks
        H, W = h, w
        reached = {}
        for bi, (c1, c2, c3, d1, d2) in enumerate(BLOCKS):
            p = f"layers.{bi + 2}.layers."
            sb = f"SB{bi + 1}"
            G = max(8, c1 // 8)
            vox = D * H * W
            # fold: its statistics input is what the producer wrote
            _, fa, fo, _ = next(it)
            n32 = -(-fa["rows"] // 32) * fa["partial_cols"] * 2
            assert _same(fa["partials"].reshape(-1)[:n32], prod["partials"].reshape(-1)[:n32]), f"{sb}: statistics partials"
            assert fa["groups"] == G and fa["eps"] == EPS and fa["cin"] == c1
            _check_stats(cs, sb + ".fold", prod, fa, fo["ab"], G, EPS)
            del prod
            layout, coutp = fa["layout"], fa["cout_pad"]
            w1 = sd[p + "1.weight"]
            bsh = _check_fold(cs, sb + ".fold", fa, fo, w1, layout, coutp)

            # convolution after the fold: raw input x folded weights + bias + the independently computed shift
            na, ca, co_, _ = next(it)
            assert _same(ca["x"], cur), f"{sb}a input"
            wimg = ca["w_taps"] if na == "conv3d_dilated_tab" else ca["w_img"]
            assert _same(wimg.reshape(-1), fo["w_out"]) and _same(ca["table"], fo["table"]), f"{sb}a operands"
            assert ca["dil"] == d1
            if na == "conv3d_dilated_tab":
                wf = _taps_from_image(fo["w_out"], c2, c1).to(F64)
            else:  # the image is bf16(w * a) laid out by rowsn_weight_image (checked bit for bit by _check_fold)
                wf = (w1 * fo["ab"][:c1].cpu().view(1, c1, 1, 1, 1)).to(BF16).to(DEV, F64)
            w64, bias = w1.to(DEV, F64), fa["bias"][:c2].to(F64)
            x64 = cur.to(F64)
            shift = _conv64(bsh, w64, d1, shape=(D, H, W))
            pre = _conv64(x64, wf, d1) + bias + shift
            S = _conv64(x64.abs(), wf.abs(), d1) + bias.abs() + _conv64(bsh.abs(), w64.abs(), d1, shape=(D, H, W))
            got = co_["out"]
            ref, bound = cs.check(sb + "a", na + " (folded)", got, pre, S, gelu=True)
            del S, ref
            rr = _rows_reached(D, H, W, d1)
            reached[sb] = rr
            interior = w64.sum((2, 3, 4)) @ bsh  # the all-taps-inside shift: what padding the RAW tensor would add
            ar = lambda n_: torch.arange(n_, device=DEV)  # noqa: E731
            borders = {"depth": ((ar(D) < d1) | (ar(D) + d1 >= D))[:, None, None],
                       "height": ((ar(H) < 1) | (ar(H) + 1 >= H))[None, :, None],
                       "width": ((ar(W) < 1) | (ar(W) + 1 >= W))[None, None, :]}
            for axis, m in borders.items():
                m = m.expand(D, H, W)[..., None]
                if bool(m.any()):
                    cs.control(sb + "a", f"table: interior row on the {axis} border", got,
                               F.gelu(torch.where(m, pre - shift + interior, pre)), bound)
            cs.conv_controls(sb + "a", got, x64, wf, pre, bound, d1)
            del pre, bound, shift, x64, got
            cur = co_["out"]

            # second convolution: plain bias
            nb, cb, cob, _ = next(it)
            assert _same(cb["x"], cur), f"{sb}b input"
            assert cb["dil"] == d2
            if nb == "conv3d_dilated":
                wb = _taps_from_image(cb["w_taps"], c2, c2).to(F64)
                bias = cb["bias"][:c2].to(F64)
            else:
                cand = sd[p + "3.weight"].to(BF16)
                assert _same(cb["w_img"], rowsn_weight_image(cand.float()).to(DEV).to(BF16)), f"{sb}b weight image"
                tab = cb["table"].view(64, c2)
                assert bool((tab == tab[:1]).all()), f"{sb}b: a plain layer's table holds its bias in every row"
                wb, bias = cand.to(DEV, F64), tab[0].to(F64)
            x64 = cur.to(F64)
            pre = _conv64(x64, wb, d2) + bias
            S = _conv64(x64.abs(), wb.abs(), d2) + bias.abs()
            got = cob["out"]
            ref, bound = cs.check(sb + "b", nb, got, pre, S, gelu=True)
            del S, ref
            cs.conv_controls(sb + "b", got, x64, wb, pre, bound, d2)
            del pre, bound, x64, got
            cur = cob["out"]

            # transposed convolution (+ statistics of what it stores)
            nt, ta, to, ret = next(it)
            assert _same(ta["x"], cur), f"{sb}.convT input"
            pre, S = _linear64(ta["x"].reshape(vox, c2), ta["w_sub"], ta["bias4"])
            # out[d, 2h + i, 2w + j, co] = column (i*2 + j) * c3 + co of input voxel (d, h, w)
            got = to["out"].view(D, H, 2, W, 2, c3).permute(0, 1, 3, 2, 4, 5).reshape(vox, 4 * c3)
            ref, _ = cs.check(sb + ".convT", nt, got, pre, S, gelu=True)
            if nt == "convT_1x2x2_gn":
                cpg = ta["cpg"]
                direct = ret[0] != vox  # register-resident sums: (32 R, 8 cpg), one partials row per epilogue thread
                n_grp = 4 * vox * cpg
                n_acc = max(4 * -(-n_grp // (ret[0] // 32)), 256) if direct else 32 * cpg
                prod = {"y": ref.view(vox, 4, c3), "B": (GELU_LIP * ACC * S + G_ERR).view(vox, 4, c3),
                        "partials": to["partials"], "n_acc": n_acc}
                print(f"  {sb}.convT statistics: {'gn_direct, ' + str(ret[0] // 32) + ' rows' if direct else 'per 32-row block'}, "
                      f"{n_acc} fp32 terms per partial sum in the bound")
            del pre, S, ref, got
            cur = to["out"]
            H, W = 2 * H, 2 * W

        # -------------------------------------------------------------- output layers
        n8, ra, ro, _ = next(it)
        assert _same(ra["x"], cur), "output_layer.0 input"
        w_o1 = sd["output_layer.0.weight"].to(BF16)
        assert _same(ra["w_img"], rows8_weight_image(w_o1.float()).to(DEV).to(BF16)), "output_layer.0 weight image"
        w64, bias = w_o1.to(DEV, F64), ra["bias8"].to(F64)
        x64 = cur.to(F64)
        pre = _conv64(x64, w64, 1) + bias
        S = _conv64(x64.abs(), w64.abs(), 1) + bias.abs()
        got = ro["out"]
        ref, bound = cs.check("out0", n8, got, pre, S, gelu=True)
        del S, ref
        cs.conv_controls("out0", got, x64, w64, pre, bound, 1)
        del pre, bound, x64, got
        cur = ro["out"]

        nf, fa_, fo_, _ = next(it)
        assert _same(fa_["x"], cur), "output_layer.2 input"
        w_o2 = sd["output_layer.2.weight"].to(BF16)
        assert _same(fa_["w_img"], rows8_weight_image(w_o2.float()).to(DEV).to(BF16)), "output_layer.2 weight image"
        w64, bias = w_o2.to(DEV, F64), fa_["bias1"].to(F64)
        x64 = cur.to(F64)
        pre = (_conv64(x64, w64, 1) + bias)[..., 0]
        bound = ACC * (_conv64(x64.abs(), w64.abs(), 1) + bias.abs())[..., 0]
        lg, pr = fo_["logits"], fo_["probs"]
        assert _same(lg, logits) and _same(pr, probs), "segment_volume returns what the last launch wrote"
        ref = pre.clamp(-5.0, 5.0)
        err = lg.to(F64) - ref
        cs.rows.append(("out2", nf + " logits", (err.abs() / bound).max().item(), (err.mean() / ref.square().mean().sqrt()).item()))
        beyond = pre.abs() > 5.0 + bound
        clipped = beyond.to(F64).mean().item()
        assert torch.equal(lg[beyond], torch.sign(pre[beyond]).float() * 5.0), "logits beyond the clip must be exactly +-5"
        perr = (pr.to(F64) - torch.sigmoid(lg.to(F64))).abs().max().item()
        cs.rows.append(("out2", nf + " probs", perr / PROB_ABS, float("nan")))
        cs.conv_controls("out2", lg[..., None], x64, w64, pre[..., None], bound[..., None], 1, gelu=False, clip=True)
        del pre, bound, x64, err, ref
    assert next(it, None) is None

    torch.cuda.synchronize()
    ref_s, ref_gb = time.perf_counter() - t_ref, (torch.cuda.max_memory_allocated() - base) / 2 ** 30

    # ------------------------------------------------------------------ report
    print(f"  {'launch':14s} {'kind':32s} {'err/bound':>10s} {'mean/rms':>10s}")
    for label, kind, r, m in cs.rows:
        print(f"  {label:14s} {kind:32s} {r:10.3f} {m:10.2e}")
    print(f"  table rows reached (from coordinates): " + ", ".join(f"{k} {len(v)}" for k, v in reached.items()))
    asserted = [x for x in cs.controls if (case, x[1]) not in PRINT_ONLY]
    printed = [x for x in cs.controls if (case, x[1]) in PRINT_ONLY]
    weakest = {}
    for label, edit, m in asserted:
        weakest[edit] = min(weakest.get(edit, float("inf")), m)
    print(f"[head-inference {case}] controls: {sum(x[2] > 1 for x in asserted)} of {len(asserted)} asserted edits break their "
          f"bounds; weakest per edit: " + ", ".join(f"{k} x{v:.3g}" for k, v in weakest.items()))
    if printed:
        print("  printed only: " + ", ".join(f"{lb} {e} x{m:.3g}" for lb, e, m in printed))
    print(f"[head-inference {case}] {100 * clipped:.1f} % of the logits beyond the clip; worst error / bound "
          f"{max(r[2] for r in cs.rows):.3f}; float64 references {ref_s:.1f} s, peak {ref_gb:.1f} GB above the recording; "
          f"{time.perf_counter() - t_case:.1f} s in all")

    # ------------------------------------------------------------------ assertions
    every = {(dm * 4 + hm) * 4 + wm for dm in (1, 2, 3) for hm in (1, 2, 3) for wm in (1, 2, 3)}
    if case == "production":  # every mask but "both taps outside" on every axis, in every folded layer
        assert all(v == every for v in reached.values()), reached
    if case == "shallow":  # D <= 24: SB1 only in dm = 0; SB2 (d = 16): dm 0, 1 (upper tap outside) and 2 (lower tap outside)
        assert {m >> 4 for m in reached["SB1"]} == {0} and {m >> 4 for m in reached["SB2"]} == {0, 1, 2}, reached
    if case == "one_row":  # H = 1 at SB1: both height taps outside
        assert {(m >> 2) & 3 for m in reached["SB1"]} == {0}, reached
    assert 0.2 <= clipped <= 0.4, clipped
    bad = [r for r in cs.rows if not r[2] <= 1.0]
    assert not bad, bad
    bad_mean = [r for r in cs.rows if r[3] == r[3] and not abs(r[3]) <= MEAN_REL]
    assert not bad_mean, bad_mean
    missed = [x for x in asserted if not x[2] > 1.0]
    assert not missed, missed
