"""Every path of the attention kernels against float64, closely enough to see one key.

``test_gpu_kernels.py::test_attention*`` compares the kernels with SDPA elementwise (atol 2e-2 x scale, rtol 2e-2). At
score std 1 an output element is an average of ~1000 values of v with magnitude 0.05-0.1, so that tolerance is 20-40 %
of it, and at large score spreads one or two keys decide each row. A padding key counted in the row sum, one key
dropped from a full tile or a SPLIT merge that ignores the partial maxima passes it. Here:

- Reference: ``softmax(q k^T / 8) v`` in float64 on the 16-bit q/k/v the kernel reads.
- Yardstick: the same with the kernel's roundings: P rounded to the operand format (bf16, or fp16 with
  ``CVIT_FMT_OPERANDS_F16``), the row sum taken from the unrounded P, the output rounded to the output format (bf16,
  fp16 or TF32 ``rna``). The ``mma.sync`` kernel (``csrc/attention.cu``) rounds the same way: bf16 P, an fp32 row sum
  of the unrounded exponentials, a bf16 output.
- Statistics against the reference, for the kernel and for the yardstick, separately over the rows of the SPLIT query
  tile and over all other rows: (a) the per-row relative error ||o - ref|| / ||ref||, its RMS and its maximum; (b) the
  per-row scale bias alpha = <o, ref> / <ref, ref> - 1 averaged over the rows. Rounding noise averages out of (b); an
  error in the denominator (padding keys in the row sum, a wrong merge normalisation, a lost rescale) shifts every row
  the same way, so (b) resolves it far below the per-row noise.
- Bounds (``_bounds``): the kernel's RMS and maximum of (a) at most ``K_RMS`` / ``K_MAX`` times the yardstick's; its
  |mean alpha| at most ``A_K`` times the yardstick's plus ``A_Z`` standard errors of the yardstick's mean.

The cases (``SHAPES``) reach every item kind (PAIRED, SPLIT, SOLO) and every ragged-tile branch (none, the short
N = 16 tile, 16-column chunks); ``_structure`` restates the kernel's item and tile logic from its own tile sizes and the
cases assert what each one reaches. The scores are shaped through one channel (q[..., 0] = 8, k[key, 0] = the key's
bias, ``_regimes``): random spreads, asymmetric SPLIT halves, maxima growing along the walked order so that the lazy
rescale fires on every tile, every second or every third, decreasing maxima where it never fires, and the whole support
in the ragged tile or in one full tile. The controls (unmarked, CPU) inject into the float64 reference one error of the
kind a rework of the kernel makes and check that it breaks the bounds by at least 2x wherever it changes the result.
The exact tests check what no tolerance sees: a slice alone and inside 16 slices, permuted heads, and the bytes around
the output.

Measured on one NVIDIA B200 (1000 W power limit), worst kernel / yardstick ratio over all cases and regimes, (a) RMS
and (a) max: bf16>bf16 1.28 and 1.56, bf16>f16 1.69 and 1.78, bf16>tf32 1.69 and 1.78, f16>f16 1.18 and 1.55,
mma.sync 1.03 and 1.08. The tcgen05 arms lose most at score std 2.5, where one or two keys carry each row and the
yardstick rounds nothing of them (``K_RMS``). Worst |mean alpha| in units of the yardstick's |mean alpha| plus one
standard error: 6.9 (bf16>bf16, T = 133), 5.6 (bf16>f16 and bf16>tf32), 11.2 (f16>f16, B 8 H 24 T 1029, where
it is 2.0e-6 against a standard error of 1.3e-7), 1.3 (mma.sync); the worst |mean alpha| is 0.63 of its bound. The
GPU tests of this file take about 8 s on that card, the controls about 14 s on a CPU.
"""
import math
import re
import time
from pathlib import Path

import pytest
import torch

from quant_emulation import rnd

F64, BF16, F16, F32 = torch.float64, torch.bfloat16, torch.float16, torch.float32
DEV = "cuda"
SRC = Path(__file__).resolve().parent.parent / "cryovit_b200" / "csrc" / "attention_tcgen05.cu"


def _kernel_constants() -> tuple[int, int, float, float]:
    """Query and key tile sizes and the lazy-rescale thresholds (log2, fp16 and bf16 probabilities), read from the
    kernel source so that a change there moves the cases' assertions with it."""
    src = SRC.read_text()
    tiles = re.search(r"constexpr int FA_BQ = (\d+), FA_BK = (\d+)", src)
    thr = re.search(r"FA_RESCALE_LOG2 = F16 \? ([\d.]+)f : ([\d.]+)f", src)
    assert tiles and thr, "tile sizes / rescale thresholds not found in attention_tcgen05.cu"
    return int(tiles[1]), int(tiles[2]), float(thr[1]), float(thr[2])


BQ, BK, RESCALE_LOG2_F16, RESCALE_LOG2_BF16 = _kernel_constants()

# Bounds, from the worst ratios measured on a B200 (module docstring) with room to spare. The kernel normalises its
# probabilities to a running maximum that lags the row's, so it rounds the P of a row's dominant key where the
# yardstick's is exactly 1: its per-row alpha scatters more, and rows that share a dominant key scatter together. The
# bias bound therefore allows A_Z standard errors of the yardstick's mean alpha plus ALPHA_FLOOR.
K_RMS = 2.5
K_MAX = 3.0
A_K = 2.0
A_Z = 16.0
ALPHA_FLOOR = 1e-5
EPS = 1e-6


# T: item kinds, ragged-tile branch ("short": the N = 16 tile in registers, "chunked": 16-column chunks, None: no
# ragged tile) and the keys of the ragged tile.
SHAPES = {
    16: ({"SOLO"}, "short", 16),           # exactly 16 keys, no padding
    29: ({"SOLO"}, "chunked", 29),
    128: ({"SOLO"}, None, 128),
    133: ({"PAIRED"}, "short", 5),         # group B's query tile has 5 rows
    256: ({"PAIRED"}, None, 128),
    257: ({"PAIRED", "SPLIT"}, "short", 1),
    261: ({"PAIRED", "SPLIT"}, "short", 5),  # three K/V tiles
    272: ({"PAIRED", "SPLIT"}, "short", 16),
    300: ({"PAIRED", "SPLIT"}, "chunked", 44),
    383: ({"PAIRED", "SPLIT"}, "chunked", 127),
    384: ({"PAIRED", "SPLIT"}, None, 128),
    789: ({"PAIRED", "SPLIT"}, "chunked", 21),
    1029: ({"PAIRED", "SPLIT"}, "short", 5),   # the production slice: 1 + 4 + 37 x 37 tokens
    1374: ({"PAIRED", "SPLIT"}, "chunked", 94),  # a 518 x 518 slice
    2121: ({"PAIRED", "SPLIT"}, "chunked", 73),  # a 644 x 644 slice: 17 query tiles
}
B_SHAPE, H_SHAPE = 2, 2
MANY_ITEMS = [(16, 8, 261), (8, 24, 1029)]  # more items than SMs: one CTA runs items of different kinds in a row

# name: (qkv dtype, output dtype, P format, output format, legacy mma.sync kernel); formats as in quant_emulation.rnd
ARMS = {
    "bf16>bf16": (BF16, BF16, "b", "b", False),
    "bf16>f16": (BF16, F16, "b", "h", False),
    "bf16>tf32": (BF16, F32, "b", "t", False),
    "f16>f16": (F16, F16, "h", "h", False),
    "mma.sync": (BF16, BF16, "b", "b", True),
}


def _structure(T: int) -> dict:
    """The kernel's work decomposition of a slice of T tokens (attention_tcgen05.cu: kv_tile, pair_kind)."""
    n_tiles, n_qt = -(-T // BK), -(-T // BQ)
    ragged = T % BK != 0
    valid = T - (n_tiles - 1) * BK
    walked = [n_tiles - 1] + list(range(n_tiles - 1)) if ragged else list(range(n_tiles))
    kinds = {"PAIRED" if 2 * p + 1 < n_qt else "SPLIT" if n_tiles > 1 else "SOLO" for p in range((n_qt + 1) // 2)}
    pos = torch.empty(T, dtype=torch.long)  # walked position of each key's tile
    for j, t in enumerate(walked):
        pos[t * BK:(t + 1) * BK] = j
    return {
        "n_tiles": n_tiles, "n_qt": n_qt, "valid": valid, "walked": walked, "kinds": kinds, "pos": pos,
        "branch": None if not ragged else "short" if valid <= 16 else "chunked",
        "pad": (-valid) % 16,  # zero-filled keys inside the ragged tile's MMA
        "split_rows": (n_qt - 1) * BQ if "SPLIT" in kinds else T,  # first row of the SPLIT query tile
        "last_tile_rows": T - (n_qt - 1) * BQ,
    }


# ------------------------------------------------------------------------------------------------ score regimes

def _regimes(T: int, pfmt: str) -> dict:
    """name -> (std of the random part of the scores, bias of each key in score units) for the regimes a slice of T
    tokens can show. The growing-maxima steps straddle the lazy-rescale threshold of the probability format
    (16 / log2 e = 11.1 score units for bf16, 8 / log2 e = 5.5 for fp16)."""
    st = _structure(T)
    pos = st["pos"].to(F64)
    zero = torch.zeros(T, dtype=F64)
    r = {f"random {s}": (s, zero) for s in (0.5, 1.0, 2.5)}
    if "SPLIT" in st["kinds"]:
        for d in (30.0, -30.0, 8.0):  # group A's tiles (walked even) against group B's (walked odd)
            r[f"split {d:+g}"] = (1.0, torch.where(pos % 2 == 0, d, 0.0))
    if st["n_tiles"] > 1:
        for g in (12.0, 10.0, 5.0, -12.0) if pfmt == "b" else (6.0, 3.0, -6.0):
            r[f"grow {g:+g}"] = (0.5, g * pos)
        if st["branch"] is not None:
            r["support ragged"] = (1.0, torch.where(pos == 0, 0.0, -60.0))
        r["support last"] = (1.0, torch.where(pos == st["n_tiles"] - 1, 0.0, -60.0))
    return r


def _qkv(B: int, T: int, H: int, sigma: float, bias: torch.Tensor, dtype, seed: int = 0) -> torch.Tensor:
    """(B, T, 3, H, 64) 16-bit q/k/v: v ~ N(0, 1); q[..., 0] = 8 and k[..., 0] = bias, so each key's score is shifted
    by its bias; the other 63 channels of q and k give random scores of std sigma."""
    g = torch.Generator().manual_seed(seed + 1000 * T + B)
    x = torch.randn(B, T, 3, H, 64, generator=g)
    x[:, :, :2] *= math.sqrt(8 * sigma / math.sqrt(63))
    x[:, :, 0, :, 0] = 8.0
    x[:, :, 1, :, 0] = bias.float()[None, :, None]
    return x.to(dtype)


# ------------------------------------------------------------------------------------------------ reference, yardstick

class _Exact:
    """float64 softmax(q k^T / 8) v of (B, T, 3, H, 64) q/k/v, with the pieces the controls edit."""

    def __init__(self, qkv: torch.Tensor):
        self.q, self.k, self.v = qkv.to(F64).permute(2, 0, 3, 1, 4)  # (B, H, T, 64)
        self.s = self.q @ self.k.transpose(-1, -2) / 8
        self.M = self.s.amax(-1, keepdim=True)
        self.e = torch.exp(self.s - self.M)
        self.l = self.e.sum(-1, keepdim=True)
        self.num = self.e @ self.v
        self.ref = self.num / self.l

    def yardstick(self, pfmt: str, ofmt: str) -> torch.Tensor:
        return rnd((rnd(self.e, pfmt).to(F64) @ self.v) / self.l, ofmt).to(F64)


def _stats(o: torch.Tensor, ref: torch.Tensor, split_row: int) -> dict:
    """(B, H, T, 64) -> {row group: (RMS and max of the per-row relative error, mean alpha, its standard error)}."""
    d = (o - ref).norm(dim=-1) / ref.norm(dim=-1)
    a = (o * ref).sum(-1) / (ref * ref).sum(-1) - 1
    out = {}
    for name, sl in (("rest", slice(0, split_row)), ("split", slice(split_row, None))):
        dd, aa = d[..., sl].flatten(), a[..., sl].flatten()
        if dd.numel():
            se = aa.std().item() / math.sqrt(aa.numel()) if aa.numel() > 1 else abs(aa.item())
            out[name] = (dd.pow(2).mean().sqrt().item(), dd.max().item(), aa.mean().item(), se)
    return out


def _bounds(y: tuple) -> tuple:
    """(a) RMS, (a) max, |(b)| bounds from the yardstick's statistics; (a) never below EPS: where one key carries a
    row, the 16-bit v it returns is exact and so is the yardstick."""
    return K_RMS * y[0] + EPS, K_MAX * y[1] + EPS, A_K * abs(y[2]) + A_Z * y[3] + ALPHA_FLOOR


def _excess(x: tuple, b: tuple) -> float:
    """The largest of (a) RMS / bound, (a) max / bound, |(b)| / bound; NaN counts as infinite."""
    r = max(x[0] / b[0], x[1] / b[1], abs(x[2]) / b[2])
    return float("inf") if math.isnan(r) else r


def _lazy(ex: _Exact, st: dict, pfmt: str):
    """The kernel's lazy-rescale decisions along the walked K/V tiles, for the rows outside the SPLIT tile: per row the
    number of rescales, the walked position of the last one and how far the running maximum jumped there (score units)."""
    thr = (RESCALE_LOG2_F16 if pfmt == "h" else RESCALE_LOG2_BF16) * math.log(2)
    s = ex.s[..., :st["split_rows"], :]
    tm = [s[..., t * BK:(t + 1) * BK].amax(-1) for t in st["walked"]]
    m = tm[0]
    count, last, jump = torch.zeros_like(m), torch.full_like(m, -1), torch.zeros_like(m)
    for j in range(1, len(tm)):
        need = tm[j] - m > thr
        last = torch.where(need, float(j), last)
        jump = torch.where(need, tm[j] - m, jump)
        count += need
        m = torch.where(need, tm[j], m)
    return count, last, jump


# ------------------------------------------------------------------------------------------------ controls

def _controls(ex: _Exact, st: dict, pfmt: str) -> dict:
    """name -> (the float64 output with one injected error, the largest share of a row's softmax weight that the keys or
    the partial it removes or adds carry, or None where the error does not remove or add weight), for each control that
    applies to this shape."""
    T, s, e, v, l, num, M = ex.s.shape[-1], ex.s, ex.e, ex.v, ex.l, ex.num, ex.M
    out = {}

    def drop(key):
        w = e[..., key:key + 1]
        return (num - w * v[..., key:key + 1, :]) / (l - w), (w / l).max().item()

    if st["branch"] is not None:
        out["drop a ragged-tile key"] = drop((st["n_tiles"] - 1) * BK + st["valid"] // 2)
    if T >= BK:
        out["drop first key of tile 0"] = drop(0)
        out["drop last key of tile 0"] = drop(BK - 1)
    out["drop the slice's last key"] = drop(T - 1)
    if st["pad"]:
        w = st["pad"] * torch.exp(-M)  # zero-filled keys: score 0, v = 0
        out["padding keys in the row sum"] = num / (l + w), (w / (l + w)).max().item()
        # the next slice's first keys where the zero fill belongs (the last slice wraps to the first)
        kn, vn = ex.k.roll(-1, 0)[..., :st["pad"], :], ex.v.roll(-1, 0)[..., :st["pad"], :]
        en = torch.exp(ex.q @ kn.transpose(-1, -2) / 8 - M)
        w = en.sum(-1, keepdim=True)
        out["next slice's keys as padding"] = (num + en @ vn) / (l + w), (w / (l + w)).max().item()
    r0 = st["split_rows"]
    if r0 < T:
        ga = (st["pos"] % 2 == 0).to(s.device, F64)  # group A's keys: walked-even tiles
        sr, er, lr = s[..., r0:, :], e[..., r0:, :], l[..., r0:, :]
        ma = sr.masked_fill(ga == 0, -math.inf).amax(-1, keepdim=True)
        mb = sr.masked_fill(ga == 1, -math.inf).amax(-1, keepdim=True)
        ea, eb = torch.exp(sr - ma) * ga, torch.exp(sr - mb) * (1 - ga)
        share_a = ((er * ga).sum(-1, keepdim=True) / lr).max().item()
        share_b = ((er * (1 - ga)).sum(-1, keepdim=True) / lr).max().item()
        for name, o_split, share in (
                ("merge ignores the partial maxima", ((ea + eb) @ v) / (ea + eb).sum(-1, keepdim=True), None),
                ("merge drops group A's partial", (eb @ v) / eb.sum(-1, keepdim=True), share_a),
                ("merge drops group B's partial", (ea @ v) / ea.sum(-1, keepdim=True), share_b)):
            o = ex.ref.clone()
            o[..., r0:, :] = o_split
            out[name] = o, share
    count, last, jump = _lazy(ex, st, pfmt)
    if count.max() > 0:  # O of the tiles before a row's last rescale keeps the old maximum's scale; l is rescaled
        pre = (st["pos"].to(s.device)[None, None, None, :] < last[..., None]).to(F64)
        o = ex.ref.clone()
        o[..., :r0, :] = (num[..., :r0, :] + (torch.exp(jump)[..., None] - 1) * ((e[..., :r0, :] * pre) @ v)) / l[..., :r0, :]
        out["one rescale of O skipped"] = o, None
    rows = st["last_tile_rows"]
    if rows >= 2:
        o = ex.ref.clone()
        a, b = T - rows, T - 1
        o[..., [a, b], :] = o[..., [b, a], :]
        out["two rows of the last query tile swapped"] = o, None
    return out


# A control that removes or adds weight is asserted where that weight reaches MIN_SHARE of some row's softmax: the
# spacing of the probability format at 1 (twice its unit roundoff). Below that (keys at -60, in tiles 10-190 below the
# row's maximum, a SPLIT partial with merge weight ~2^-43) the output may move by less than the rounding noise; such
# controls are printed when they stay within 2x of the bounds, not asserted.
MIN_SHARE = {"b": 2 ** -7, "h": 2 ** -10}


@pytest.mark.parametrize("T", list(SHAPES))
def test_controls_break_the_bounds(T):
    """Each control breaks the bounds the yardstick sets by at least 2x in every regime where what it removes or adds
    carries weight (``MIN_SHARE``); the rest are printed. The bounds depend on the yardstick alone: no GPU needed."""
    st = _structure(T)
    assert (st["kinds"], st["branch"], st["valid"]) == SHAPES[T], st
    asserted, printed = [], []
    for pfmt, ofmt in (("b", "b"), ("h", "h")):
        for regime, (sigma, bias) in _regimes(T, pfmt).items():
            ex = _Exact(_qkv(B_SHAPE, T, H_SHAPE, sigma, bias, BF16 if pfmt == "b" else F16))
            if regime.startswith("grow"):  # decreasing maxima never rescale; growing ones do once they outgrow the threshold
                rescales = _lazy(ex, st, pfmt)[0].max().item()
                g, thr = float(regime.split()[1]), (RESCALE_LOG2_F16 if pfmt == "h" else RESCALE_LOG2_BF16) * math.log(2)
                assert rescales == 0 if g < 0 else rescales > 0 or g * (st["n_tiles"] - 1) < thr + 3, (regime, rescales)
            y = _stats(ex.yardstick(pfmt, ofmt), ex.ref, st["split_rows"])
            for name, (o, share) in _controls(ex, st, pfmt).items():
                c = _stats(o, ex.ref, st["split_rows"])
                x = max(_excess(c[g], _bounds(y[g])) for g in c)
                (asserted if share is None or share >= MIN_SHARE[pfmt] else printed).append((pfmt, regime, name, share, x))
    print(f"\n[attention controls T={T}] {len(asserted)} asserted, the weakest x{min(a[4] for a in asserted):.1f}; "
          f"{len(printed)} where the control carries less weight, within 2x of the bounds in these regimes:")
    for name in dict.fromkeys(a[2] for a in printed):
        within = [f"{p} {reg} x{x:.2f}" for p, reg, n, share, x in printed if n == name and x < 2]
        if within:
            print(f"  {name}: " + ", ".join(within))
    missed = [a for a in asserted if not a[4] >= 2]
    assert not missed, missed


# ------------------------------------------------------------------------------------------------ GPU

def _launch(qkv: torch.Tensor, arm: str, out: torch.Tensor | None = None) -> torch.Tensor:
    """Run one arm on (B, T, 3, H, 64) q/k/v; returns the (B*T, H*64) output (NaN-filled before the launch)."""
    from cryovit_b200 import ops

    qd, od, _, _, legacy = ARMS[arm]
    B, T, _, H, _ = qkv.shape
    x = qkv.to(DEV, qd).reshape(B * T, 3 * H * 64).contiguous()
    if out is None:
        out = torch.full((B * T, H * 64), float("nan"), device=DEV, dtype=od)
    ops.attention(x, out, B, T, H, legacy_mma_sync=legacy)
    return out


def _parity(B: int, T: int, H: int, regimes: list | None = None) -> list:
    """Every arm in every regime of the shape against float64; returns rows (arm, regime, row group, kernel stats,
    yardstick stats, excess over the bounds)."""
    st = _structure(T)
    rows = []
    for qd in (BF16, F16):
        pfmt = "b" if qd == BF16 else "h"
        arms = [a for a, c in ARMS.items() if c[0] == qd]
        for regime, (sigma, bias) in _regimes(T, pfmt).items():
            if regimes is not None and regime not in regimes:
                continue
            qkv = _qkv(B, T, H, sigma, bias, qd).to(DEV)
            ex = _Exact(qkv)
            for arm in arms:
                _, _, pf, of, _ = ARMS[arm]
                y = _stats(ex.yardstick(pf, of), ex.ref, st["split_rows"])
                out = _launch(qkv, arm)
                assert not out.isnan().any(), f"{arm} {regime}: output elements not written"
                o = out.view(B, T, H, 64).permute(0, 2, 1, 3).to(F64)
                k = _stats(o, ex.ref, st["split_rows"])
                for g in k:
                    rows.append((arm, regime, g, k[g], y[g], _excess(k[g], _bounds(y[g]))))
            del ex
    return rows


def _report(tag: str, rows: list) -> None:
    """Per arm: the worst kernel / yardstick ratio of (a) RMS, (a) max and (b) |alpha| in units of the yardstick's bias
    plus its standard error, the worst |alpha| over its bound, and the worst excess over the bounds with its regime."""
    for arm in ARMS:
        mine = [r for r in rows if r[0] == arm]
        if not mine:
            continue
        w = max(mine, key=lambda r: r[5])
        rr = max(r[3][0] / r[4][0] for r in mine if r[4][0] > 0)
        rm = max(r[3][1] / r[4][1] for r in mine if r[4][1] > 0)
        ra = max(abs(r[3][2]) / (abs(r[4][2]) + r[4][3]) for r in mine if r[4][3] > 0)
        rb = max(abs(r[3][2]) / _bounds(r[4])[2] for r in mine)
        print(f"[attention parity {tag}] {arm:9s} worst RMS ratio {rr:.2f}, max ratio {rm:.2f}, |alpha| / (|alpha_y| + se_y) "
              f"{ra:.2f}, |alpha| / bound {rb:.2f}; worst excess {w[5]:.2f} ({w[1]}, {w[2]} rows: RMS {w[3][0]:.2e} max {w[3][1]:.2e} "
              f"alpha {w[3][2]:+.1e} against {w[4][0]:.2e} {w[4][1]:.2e} {w[4][2]:+.1e} se {w[4][3]:.1e})")


@pytest.mark.gpu
@pytest.mark.parametrize("T", list(SHAPES))
def test_attention_matches_float64(cuda_lib, T):
    st = _structure(T)
    assert (st["kinds"], st["branch"], st["valid"]) == SHAPES[T], st
    t0 = time.perf_counter()
    rows = _parity(B_SHAPE, T, H_SHAPE)
    _report(f"T={T}", rows)
    print(f"[attention parity T={T}] {len(rows)} comparisons, {time.perf_counter() - t0:.1f} s")
    bad = [r[:3] + (round(r[5], 2),) for r in rows if not r[5] <= 1]
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,T", MANY_ITEMS)
def test_attention_matches_float64_many_items(cuda_lib, B, H, T):
    """More items than SMs, so that one CTA runs items of different kinds one after another."""
    st = _structure(T)
    items = (st["n_qt"] + 1) // 2 * H * B
    assert items > torch.cuda.get_device_properties(0).multi_processor_count and "SPLIT" in st["kinds"], items
    rows = _parity(B, T, H, ["random 1.0", "split +30", "split -30", "grow +12", "grow +6"])
    _report(f"B={B} H={H} T={T}", rows)
    bad = [r[:3] + (round(r[5], 2),) for r in rows if not r[5] <= 1]
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("arm", list(ARMS))
def test_attention_slice_alone_equals_slice_in_batch(cuda_lib, arm):
    """A slice computed alone and as slice 11 of a 16-slice launch is bit-identical, at every T: barrier phases, the
    item parity of the group barriers across item kinds, stale TMEM O / P and the grid-stride order leak into neither."""
    qd = ARMS[arm][0]
    for T in SHAPES:
        qkv = _qkv(16, T, H_SHAPE, 1.0, torch.zeros(T, dtype=F64), qd).to(DEV)
        whole = _launch(qkv, arm).view(16, T, -1)
        alone = _launch(qkv[11:12].contiguous(), arm).view(1, T, -1)
        assert torch.equal(whole[11].view(torch.uint8), alone[0].view(torch.uint8)), (arm, T)


@pytest.mark.gpu
@pytest.mark.parametrize("arm", list(ARMS))
def test_attention_head_permutation(cuda_lib, arm):
    """Permuting the heads of qkv permutes the output's head columns, bit for bit."""
    qd = ARMS[arm][0]
    for B, T, H in ((2, 1029, 6), (3, 261, 5), (1, 2121, 3)):
        qkv = _qkv(B, T, H, 1.0, torch.zeros(T, dtype=F64), qd).to(DEV)
        perm = torch.randperm(H, generator=torch.Generator().manual_seed(T)).to(DEV)
        out = _launch(qkv, arm).view(B, T, H, 64)
        outp = _launch(qkv[:, :, :, perm].contiguous(), arm).view(B, T, H, 64)
        assert torch.equal(outp.view(torch.uint8), out[:, :, perm].view(torch.uint8)), (arm, B, T, H)


@pytest.mark.gpu
@pytest.mark.parametrize("arm", list(ARMS))
def test_attention_guard_bands(cuda_lib, arm):
    """The output sits inside a larger buffer filled with a sentinel: every element of it is written, the tail tokens
    of the last slice included, and no byte before or after it changes."""
    od = ARMS[arm][1]
    guard = 4096  # elements on either side (a multiple of 16 bytes: the kernels store 16-byte vectors)
    for T in SHAPES:
        B, H = 3, 2
        qkv = _qkv(B, T, H, 1.0, torch.zeros(T, dtype=F64), ARMS[arm][0]).to(DEV)
        n = B * T * H * 64
        buf = torch.empty(n + 2 * guard, device=DEV, dtype=od)
        buf.view(torch.uint8).fill_(0xFF)  # NaN in every format: the kernels never write one
        sentinel = buf[:guard].clone()
        _launch(qkv, arm, out=buf[guard:guard + n].view(B * T, H * 64))
        assert torch.equal(buf[:guard].view(torch.uint8), sentinel.view(torch.uint8)), (arm, T, "before")
        assert torch.equal(buf[guard + n:].view(torch.uint8), sentinel.view(torch.uint8)), (arm, T, "after")
        unwritten = buf[guard:guard + n].view(B * T, -1).isnan().any(-1).nonzero()
        assert unwritten.numel() == 0, (arm, T, "rows not written", unwritten[:8].flatten().tolist())
