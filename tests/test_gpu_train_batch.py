"""A training step on a batch of crops (``CryoVITHeadTrainerB200.train_batch``, ``datamodule.dataloader.batch_size``)
against a float64 autograd restatement of the reference: ``collate_fn``'s padded batch through the head, the masked
Dice loss of the whole batch (``oracle.metrics.masked_select`` / ``dice_loss``), one backward.

The tolerance rule is ``test_gpu_train_parity.py``'s: the same float64 graph run again with every tensor the trainer
stores in bf16 rounded to bf16 is the yardstick, and every gradient piece (a 3x3x3 tap, a 1x2x2 sub-pixel, else the
whole tensor) of the trainer may be at most ``K`` times as far from float64 (``_bound``). Two controls must fail that
bound: the mean of the two crops' separate gradients (a per-crop Dice) and the batch gradient with the short crop run
unpadded (padding ignored). Then: a batch of one is the single-crop step bit for bit, seeded batch runs repeat bit for
bit, a replayed batch graph is the eager step, and the entry point trains with ``batch_size=2``.

Measured on one B200 (1000 W power limit): worst error / bound 0.59 (production plane, depths 40 and 33) and 0.63 (384
channels, 16x12, depths 36 and 29); loss error / yardstick 0.94 and 0.85. The controls miss their bounds by x7.1 (mean of
per-crop gradients) and x6.7 (short crop unpadded) on the production plane, x7.9 and x7.8 on the other. The float64
restatement is within 7e-7 of ``oracle.head.forward`` (float32, TF32 off) in every probability."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
DEV = "cuda"
F64, BF16 = torch.float64, torch.bfloat16

# test_gpu_train_parity.py's rule, restated here
K = 4.0
NOISE_K = 2.0
FLOOR = 5e-3
CAP = 5e-2
LOSS_FLOOR = 1e-6

# two crops of different depths per case, at depths the dilations reach; C, plane, feature dtype
CASES = {
    "production plane": dict(C=1536, depths=(40, 33), h=32, w=32),
    "384 channels, non-square plane": dict(C=384, depths=(36, 29), h=16, w=12),
}


def _bound(y: float) -> float:
    return max(min(K * y, CAP), NOISE_K * y, FLOOR)


def _pieces(g: torch.Tensor) -> dict:
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
    n = ref.norm().item()
    d = (got.to(F64) - ref).norm().item()
    return d / n if n > 0 else (0.0 if d == 0 else float("inf"))


def _worst(got: dict, ref: dict, yard: dict) -> tuple[float, str]:
    """The largest error / bound over every piece of every parameter, and where."""
    worst, where = 0.0, ""
    for k in ref:
        pr, pg, py = _pieces(ref[k]), _pieces(got[k]), _pieces(yard[k])
        for n in pr:
            r = _rel(pg[n], pr[n]) / _bound(_rel(py[n], pr[n]))
            if r > worst:
                worst, where = r, f"{k} {n}"
    return worst, where


class _Store(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, fwd: bool, bwd: bool):
        ctx.bwd = bwd
        return x.to(BF16).to(x.dtype) if fwd else x.clone()

    @staticmethod
    def backward(ctx, g):
        return (g.to(BF16).to(g.dtype) if ctx.bwd else g), None, None


def _head(P: dict, x: torch.Tensor, bf16: bool) -> torch.Tensor:
    """oracle.head.forward_volume's graph in float64 with autograd: x (B, C, D, h, w) -> clipped logits (B, D, 16h, 16w).
    ``bf16``: every activation, activation gradient and weight operand the trainer keeps in bf16 rounded to bf16 (the
    projection weight of the fp16 channels-first path to fp16)."""
    from cryovit_b200.head import BLOCKS

    if bf16:
        st = lambda t: _Store.apply(t, True, True)  # noqa: E731
        grad_only = lambda t: _Store.apply(t, False, True)  # noqa: E731
        wt = lambda t, dt=BF16: t + (t.detach().to(dt).to(F64) - t.detach())  # noqa: E731
    else:
        st = grad_only = wt = lambda t, *_: t  # noqa: E731
    x = st(F.gelu(st(F.conv3d(x, wt(P["layers.0.weight"], torch.float16), P["layers.0.bias"]))))
    for bi, (c1, c2, c3, d1, d2) in enumerate(BLOCKS):
        p = f"layers.{bi + 2}.layers."
        x = st(F.group_norm(x, max(8, c1 // 8), P[p + "0.weight"], P[p + "0.bias"], 1e-3))
        x = st(F.gelu(st(F.conv3d(x, wt(P[p + "1.weight"]), P[p + "1.bias"], padding="same", dilation=(d1, 1, 1)))))
        x = st(F.gelu(st(F.conv3d(x, wt(P[p + "3.weight"]), P[p + "3.bias"], padding="same", dilation=(d2, 1, 1)))))
        x = st(F.gelu(st(F.conv_transpose3d(x, wt(P[p + "5.weight"]), P[p + "5.bias"], stride=(1, 2, 2)))))
    x = st(F.gelu(st(F.conv3d(x, wt(P["output_layer.0.weight"]), P["output_layer.0.bias"], padding="same"))))
    return torch.clip(grad_only(F.conv3d(x, wt(P["output_layer.2.weight"]), P["output_layer.2.bias"], padding="same")), -5, 5)[:, 0]


def _reference(sd: dict, groups: list, bf16: bool, mean_of_groups: bool = False):
    """float64 autograd of a step. ``groups``: a list of collate_fn batches (BatchedTomogramData); one group is the batch.
    The Dice of each group is taken over all of its samples (oracle.metrics); with several groups the loss is their sum,
    or their mean with ``mean_of_groups`` (the per-crop Dice control). Returns (loss, {key: gradient})."""
    from oracle import metrics as om

    P = {k: v.to(DEV, F64).requires_grad_(True) for k, v in sd.items()}
    losses = []
    for b in groups:
        x = b.tomo_batch.permute(0, 2, 1, 3, 4).to(DEV, F64)  # collate_fn's (B, D, C, h, w) -> (B, C, D, h, w)
        probs = torch.sigmoid(_head(P, x, bf16))
        yp, yt = om.masked_select(probs, b.labels.to(DEV, F64))
        losses.append(om.dice_loss(yp, yt))
    loss = sum(losses) / (len(losses) if mean_of_groups else 1)
    loss.backward()
    return loss.item(), {k: v.grad for k, v in P.items()}


def _crops(C: int, depths, h: int, w: int, seed: int = 11):
    """Randomised GroupNorm affines, output_layer.2 scaled so that about 30 % of the logits pass the clip, fp16 feature crops
    and {0, 1} labels with ignored planes at both depth ends and scattered ignored voxels."""
    from cryovit_b200.head import BLOCKS
    from cryovit_b200.host.datasets import TomogramData
    from oracle import head as ohead

    sd = ohead.random_state_dict(C, seed=seed)
    g = torch.Generator().manual_seed(seed)
    for bi, (c1, _, _, _, _) in enumerate(BLOCKS):
        p = f"layers.{bi + 2}.layers.0."
        sd[p + "weight"] = 1.0 + 0.3 * (2 * torch.rand(c1, generator=g) - 1)
        sd[p + "bias"] = 0.5 * (2 * torch.rand(c1, generator=g) - 1)
    gd = torch.Generator(device=DEV).manual_seed(seed)
    items = []
    for i, D in enumerate(depths):
        feats = (torch.randn(C, D, h, w, generator=gd, device=DEV) * 0.5).half()
        lab = (torch.rand(D, 16 * h, 16 * w, generator=gd, device=DEV) < 0.35).float()
        lab[:2] = -1
        lab[-2:] = -1
        lab[torch.rand(D, 16 * h, 16 * w, generator=gd, device=DEV) < 0.05] = -1
        items.append(TomogramData("S", f"t{i}", None, feats, lab))
    sd_dev = {k: v.to(DEV) for k, v in sd.items()}
    logits = ohead.forward_volume(sd_dev, items[0].data.float()[None])[0, 0]
    dev = (logits - sd["output_layer.2.bias"].item()).abs().flatten()
    q = torch.quantile(dev[::max(1, dev.numel() // (1 << 22))], 0.70).item()
    sd["output_layer.2.weight"] = sd["output_layer.2.weight"] * (5.0 / q)
    return sd, items


@pytest.mark.parametrize("case", list(CASES))
def test_batch_step_gradients_match_float64_of_the_padded_batch(cuda_lib, case):
    from cryovit_b200.host.datasets import collate_fn
    from cryovit_b200.train import CryoVITHeadTrainerB200
    from oracle import head as ohead

    c = CASES[case]
    sd, items = _crops(c["C"], c["depths"], c["h"], c["w"])
    tr = CryoVITHeadTrainerB200(c["C"], state_dict=sd)
    fshape = (2, c["C"], max(c["depths"]), c["h"], c["w"])
    loss = float(tr._batch_graphed([(it.data, it.label) for it in items], fshape, torch.float16, torch.float32, 1.0))
    got = {k: tr.g[k].to(F64) for k in tr.keys}
    del tr
    torch.cuda.synchronize()
    torch.cuda.empty_cache()

    batch = collate_fn([type(it)(it.sample, it.tomo_name, None, it.data.cpu(), it.label.cpu()) for it in items])
    # the restatement is the oracle's head on collate_fn's batch (the oracle runs in float32: TF32 off for it)
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            P = {k: v.to(DEV, F64) for k, v in sd.items()}
            mine = torch.sigmoid(_head(P, batch.tomo_batch.permute(0, 2, 1, 3, 4).to(DEV, F64), False))
            oracle = ohead.forward({k: v.to(DEV) for k, v in sd.items()}, batch.tomo_batch.to(DEV))
            tie = (mine - oracle.to(F64)).abs().max().item()
            del P, mine, oracle
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    print(f"\n[train-batch {case}] float64 restatement vs oracle.head.forward (float32): max |probability difference| {tie:.2e}")
    assert tie < 1e-3
    ref_loss, ref = _reference(sd, [batch], False)
    yard_loss, yard = _reference(sd, [batch], True)
    worst, where = _worst(got, ref, yard)
    loss_err, loss_yard = abs(loss - ref_loss), abs(yard_loss - ref_loss)
    print(f"\n[train-batch {case}] depths {c['depths']}: worst error / bound {worst:.3f} ({where}); loss {loss:.7f} float64 {ref_loss:.7f} "
          f"error {loss_err:.2e} yardstick {loss_yard:.2e}")

    # controls: (a) a Dice per crop, gradients averaged; (b) the short crop run at its own depth (padding ignored)
    singles = [collate_fn([type(it)(it.sample, it.tomo_name, None, it.data.cpu(), it.label.cpu())]) for it in items]
    _, ctrl_mean = _reference(sd, singles, False, mean_of_groups=True)
    short = int(np.argmin(c["depths"]))
    # the batch-wide Dice with the short crop unpadded: its sums enter the same loss, its volume is not padded
    from oracle import metrics as om

    Pc = {k: v.to(DEV, F64).requires_grad_(True) for k, v in sd.items()}
    yps, yts = [], []
    for i, it in enumerate(items):
        x = (batch.tomo_batch[i:i + 1, :it.data.shape[1]] if i == short else batch.tomo_batch[i:i + 1]).permute(0, 2, 1, 3, 4)
        lab = batch.labels[i:i + 1, :it.data.shape[1]] if i == short else batch.labels[i:i + 1]
        yp, yt = om.masked_select(torch.sigmoid(_head(Pc, x.to(DEV, F64), False)), lab.to(DEV, F64))
        yps.append(yp)
        yts.append(yt)
    om.dice_loss(torch.cat(yps), torch.cat(yts)).backward()
    ctrl_unpadded = {k: v.grad for k, v in Pc.items()}
    miss_mean, w_mean = _worst(ctrl_mean, ref, yard)
    miss_unpadded, w_unpadded = _worst(ctrl_unpadded, ref, yard)
    print(f"[train-batch {case}] controls: mean of per-crop gradients misses its bound x{miss_mean:.2f} ({w_mean}); "
          f"short crop unpadded x{miss_unpadded:.2f} ({w_unpadded})")

    assert loss_err <= max(K * loss_yard, LOSS_FLOOR), (loss, ref_loss, yard_loss)
    assert worst <= 1.0, (worst, where)
    assert miss_mean > 1.0 and miss_unpadded > 1.0, (miss_mean, miss_unpadded)


def _det_trainer(C: int, sd: dict):
    from cryovit_b200.train import CryoVITHeadTrainerB200

    return CryoVITHeadTrainerB200(C, state_dict=sd, deterministic=True, lr=1e-3)


@pytest.fixture
def deterministic_torch():
    prev = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])


def test_batch_of_one_is_the_single_crop_step(cuda_lib, deterministic_torch, monkeypatch):
    """Three steps each (the third captured and replayed): weights, AdamW moments and losses bit for bit."""
    monkeypatch.setenv("CVIT_TRAIN_GRAPH", "1")
    sd, items = _crops(384, (36,), 16, 12)
    f, l = items[0].data, items[0].label
    a, b = _det_trainer(384, sd), _det_trainer(384, sd)
    la = [a.train_batch([(f, l)]).clone() for _ in range(3)]
    lb = [b.train_step(f, l).clone() for _ in range(3)]
    assert any("graph" in e for e in a._graphs.values()) and any("graph" in e for e in b._graphs.values())
    for t in ("flat_p", "flat_m", "flat_v", "flat_g"):
        assert torch.equal(getattr(a, t), getattr(b, t)), t
    assert all(torch.equal(x, y) for x, y in zip(la, lb)), (la, lb)


def test_replayed_batch_graph_is_the_eager_step(cuda_lib, deterministic_torch, monkeypatch):
    """Five steps on batches whose crops swap places (same Dmax, different padding): one graph, replayed with other
    padding, bit for bit the eager steps."""
    sd, items = _crops(384, (36, 29), 16, 12)
    batches = [[(it.data, it.label) for it in items], [(it.data, it.label) for it in items[::-1]]]
    runs = []
    for graph in ("0", "1"):
        monkeypatch.setenv("CVIT_TRAIN_GRAPH", graph)
        tr = _det_trainer(384, sd)
        losses = [tr.train_batch(batches[s % 2]).clone() for s in range(5)]
        runs.append((tr, losses))
    (e, le), (g, lg) = runs
    assert not e._graphs and len(g._graphs) == 1 and all("graph" in v for v in g._graphs.values())
    for t in ("flat_p", "flat_m", "flat_v", "flat_g"):
        assert torch.equal(getattr(e, t), getattr(g, t)), t
    assert all(torch.equal(x, y) for x, y in zip(le, lg))
    assert len({float(x) for x in lg}) > 1


def test_train_batch_refuses_different_feature_planes(cuda_lib):
    from cryovit_b200._lib import CryovitB200Error
    from cryovit_b200.train import CryoVITHeadTrainerB200

    tr = CryoVITHeadTrainerB200(384)
    a = (torch.zeros(384, 4, 3, 3, device=DEV, dtype=torch.float16), torch.zeros(4, 48, 48, device=DEV))
    b = (torch.zeros(384, 4, 3, 4, device=DEV, dtype=torch.float16), torch.zeros(4, 48, 64, device=DEV))
    with pytest.raises(CryovitB200Error, match=r"\(384, 4, 3, 3\) and \(384, 4, 3, 4\)"):
        tr.train_batch([a, b])
    assert tr.step_count == 0


def _toy_split(root: Path):
    from cryovit.datasets import TomoDataset
    from cryovit_b200.host import hdf

    rng = np.random.default_rng(4)
    recs = []
    for i, d in enumerate((4, 6, 5, 4, 7)):
        feats = (0.1 * rng.standard_normal((384, d, 3, 3))).astype(np.float16)
        feats[0] = 2.0 * np.sign(rng.standard_normal((d, 3, 3)))
        lab = (np.repeat(np.repeat(feats[0].astype(np.float32), 16, axis=1), 16, axis=2) > 0).astype(np.int8)
        lab[0, :8] = -1
        hdf.write_tomogram(root / "S" / f"t{i}.hdf", {"data": np.zeros((d, 48, 48), np.uint8), "labels/mito": lab, "dino_features": feats})
        recs.append({"sample": "S", "tomo_name": f"t{i}.hdf"})
    return TomoDataset(recs, "dino_features", "mito", "split_id", root, train=True)


def test_fit_head_batches_are_reproducible(cuda_lib, tmp_path):
    from cryovit_b200.host.fit import fit_head
    from oracle import head as ohead

    ds = _toy_split(tmp_path / "data")
    for tag in ("a", "b"):
        fit_head(ds, in_channels=384, max_epochs=3, lr=2e-3, swa_epoch_start=1, exp_dir=tmp_path / tag,
                 state_dict=ohead.random_state_dict(384, seed=5), deterministic=True, batch_size=2)
    wa, wb = (torch.load(tmp_path / t / "weights.pt") for t in ("a", "b"))
    assert wa.keys() == wb.keys() and all(torch.equal(wa[k], wb[k]) for k in wa)
    w1 = fit_head(ds, in_channels=384, max_epochs=3, lr=2e-3, swa_epoch_start=1, state_dict=ohead.random_state_dict(384, seed=5),
                  deterministic=True, batch_size=1)
    assert any(not torch.equal(wa[k], w1[k]) for k in wa)  # batches of two are another optimisation than single crops


def test_train_model_with_batch_size_two(cuda_lib, tmp_path):
    import pandas as pd
    from cryovit_b200.host import hdf

    rng = np.random.default_rng(4)
    rows = []
    for s in ("A", "B"):
        for i in range(4):
            d = 4 + i
            feats = (0.1 * rng.standard_normal((384, d, 3, 3))).astype(np.float16)
            feats[0] = 2.0 * np.sign(rng.standard_normal((d, 3, 3)))
            lab = (np.repeat(np.repeat(feats[0].astype(np.float32), 16, axis=1), 16, axis=2) > 0).astype(np.int8)
            hdf.write_tomogram(tmp_path / "data" / "tomograms" / s / f"{s}{i}.hdf",
                               {"data": rng.integers(0, 256, (d, 48, 48), dtype=np.uint8), "labels/mito": lab, "dino_features": feats})
            rows.append((s, f"{s}{i}.hdf", i % 2))
    (tmp_path / "data" / "csv").mkdir(parents=True, exist_ok=True)
    pd.DataFrame(rows, columns=["sample", "tomo_name", "split_id"]).to_csv(tmp_path / "data" / "csv" / "splits.csv", index=False)
    env = dict(os.environ, PYTHONPATH=str(ROOT) + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "cryovit.training.train_model", "model=cryovit", "+experiments=multi_mito",
                        "datamodule.sample=[A,B]", "datamodule.split_id=0", "+model.in_channels=384", f"paths.data_dir={tmp_path / 'data'}",
                        f"paths.exp_dir={tmp_path / 'exp'}", "trainer.max_epochs=3", "datamodule.dataloader.batch_size=2"],
                       cwd=str(ROOT), env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "batch size 2" in r.stdout + r.stderr
    assert next((tmp_path / "exp").rglob("weights.pt")).exists()
    val = pd.read_csv(next((tmp_path / "exp").rglob("validation.csv")))
    assert len(val) == 3 and val["epoch"].tolist() == [0, 1, 2]
