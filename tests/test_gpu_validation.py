"""Validation during head training: the scoring epilogue of the output convolution (cvit_conv3d_rows8_score) against
the unfused path, CryoVITHeadB200.score_volume, the trainer -> inference-head weight hand-over, the validation loop
of fit_head and train_model, and the Lightning schedule rules (the last group and the ABI refusals need no GPU)."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

DEV = "cuda"
ROOT = Path(__file__).resolve().parent.parent
gpu = pytest.mark.gpu
COUNTS = [1, 3, 4, 5, 6, 7]  # the integer sums of seg_stats; 0 and 2 are the soft ones


def _close_soft(got, ref, rel=1e-6):
    for k in (0, 2):
        assert abs(float(got[k]) - float(ref[k])) <= rel * abs(float(ref[k])) + 1e-12, (k, float(got[k]), float(ref[k]))


# ----------------------------------------------------------------------------------------------- schedule (CPU)
def test_val_schedule_follows_lightning_rules():
    from cryovit_b200.host.validate import val_schedule

    assert val_schedule(1, 1.0, 10) == (1, 10)          # defaults: every epoch, every tomogram
    assert val_schedule(3, 1.0, 10) == (3, 10)
    assert val_schedule(1, 0.5, 10) == (1, 5)           # a float is a fraction
    assert val_schedule(1, 0.25, 10) == (1, 2)          # int(10 * 0.25)
    assert val_schedule(1, 4, 10) == (1, 4)             # an int is a count ...
    assert val_schedule(1, 40, 10) == (1, 10)           # ... capped at the set
    assert val_schedule(1, 0, 10) == (1, 0) and val_schedule(1, 0.0, 10) == (1, 0)  # 0 disables
    assert val_schedule(1, 1.0, 0) == (1, 0)
    for bad in ((0, 1.0), (1.5, 1.0), (True, 1.0), (1, -1), (1, 1.5), (1, "all"), (1, True)):
        with pytest.raises(ValueError):
            val_schedule(*bad, 10)
    with pytest.raises(ValueError, match="less than one"):
        val_schedule(1, 0.05, 10)                       # Lightning refuses a fraction that leaves no batch
    # epoch e is validated when (e + 1) % n == 0
    from cryovit_b200.host.validate import Validator
    from cryovit_b200.host.metrics import DiceLoss, DiceMetric, F1Metric

    v = Validator(list(range(4)), 384, {"dice_loss": DiceLoss()}, {"dice_metric": DiceMetric(), "f1_metric": F1Metric()}, 3, 1.0)
    assert [e for e in range(10) if v.scheduled(e)] == [2, 5, 8]
    assert not any(Validator(list(range(4)), 384, {}, {}, 1, 0).scheduled(e) for e in range(5))


def test_validator_refuses_unknown_losses_and_metrics():
    from cryovit_b200.host.validate import Validator

    with pytest.raises(ValueError, match="loss 'bce'"):
        Validator([0], 384, {"bce": object()}, {}, 1, 1.0)
    with pytest.raises(ValueError, match="metric 'iou'"):
        Validator([0], 384, {}, {"iou": object()}, 1, 1.0)


def test_score_abi_refusals():
    """W % 8 != 0 -> CVIT_ERR_UNSUPPORTED; null labels / partials / out8 -> CVIT_ERR_INVALID (checked before any CUDA call)."""
    from cryovit_b200 import _lib, build

    build.build()
    lib = _lib.load()
    fake = 1 << 20  # 16-byte aligned, never dereferenced: the arguments are refused first
    f = lib.cvit_conv3d_rows8_score
    assert f(fake, fake, fake, fake, 2, 16, 60, 0.5, fake, fake, None) == -4
    assert "multiple of 8" in lib.cvit_last_error().decode()
    assert f(fake, fake, fake, None, 2, 16, 64, 0.5, fake, fake, None) == -1
    assert f(fake, fake, fake, fake, 2, 16, 64, 0.5, None, fake, None) == -1
    assert f(fake, fake, fake, fake, 2, 16, 64, 0.5, fake, None, None) == -1
    assert f(None, fake, fake, fake, 2, 16, 64, 0.5, fake, fake, None) == -1
    assert lib.cvit_conv3d_rows8_score_partials(128, 512, 512) == 8 * 2 * 64 * 8


# ----------------------------------------------------------------------------------------------- the kernel
def _final_operands(seed):
    from cryovit_b200.head import rows8_weight_image

    g = torch.Generator().manual_seed(seed)
    w = (torch.rand(1, 8, 3, 3, 3, generator=g) * 2 - 1) * 0.3
    return rows8_weight_image(w).to(DEV).bfloat16(), (torch.rand(1, generator=g) - 0.5).to(DEV)


@gpu
@pytest.mark.parametrize("D", [1, 5, 37])
@pytest.mark.parametrize("HW", [(48, 48), (40, 56), (512, 512)])
def test_score_kernel_matches_final_plus_seg_stats(cuda_lib, D, HW):
    from cryovit_b200 import ops

    H, W = HW
    g = torch.Generator().manual_seed(D * 1000 + W)
    x = (torch.randn(D, H, W, 8, generator=g) * 2).to(DEV).bfloat16()
    w_img, b = _final_operands(D + W)
    probs = torch.empty(D, H, W, device=DEV)
    ops.conv3d_rows8_final(x, w_img, b, None, probs)
    part = torch.empty(ops.rows8_score_partials(D, H, W), device=DEV, dtype=torch.float64)
    r = torch.rand(D, H, W, generator=g)
    lab_rand = torch.where(r < 0.3, -1, (torch.rand(D, H, W, generator=g) < 0.5).long()).to(torch.int8)
    cases = {"random": lab_rand, "ignored": torch.full((D, H, W), -1, dtype=torch.int8), "ones": torch.ones(D, H, W, dtype=torch.int8)}
    for name, lab in cases.items():
        for thr in (0.5, 0.37):
            lab_d = lab.to(DEV)
            out = torch.empty(8, device=DEV, dtype=torch.float64)
            got = ops.conv3d_rows8_score(x, w_img, b, lab_d, part, out, thr).clone()
            ref = ops.seg_stats(probs.view(-1), lab_d.float().view(-1), thr)
            assert torch.equal(got[COUNTS], ref[COUNTS]), (name, thr, got.tolist(), ref.tolist())
            _close_soft(got, ref)
            if name == "ignored":
                assert torch.equal(got, torch.zeros(8, device=DEV, dtype=torch.float64))
            again = ops.conv3d_rows8_score(x, w_img, b, lab_d, part, torch.empty_like(out), thr)
            assert torch.equal(again, got), "two launches must give bit-identical sums"
    assert int(ref[1]) == D * H * W  # "ones": every voxel counted


# ----------------------------------------------------------------------------------------------- score_volume
def _head(C, seed=0):
    from cryovit_b200.head import CryoVITHeadB200
    from oracle import head as ohead

    return CryoVITHeadB200(C).load_state_dict(ohead.random_state_dict(C, seed=seed)).cuda()


def _labels(D, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    r = torch.rand(D, H, W, generator=g)
    return torch.where(r < 0.3, -1, (torch.rand(D, H, W, generator=g) < 0.4).long()).to(torch.int8).to(DEV)


@gpu
@pytest.mark.parametrize("C,shape", [(384, (4, 3, 5)), (1536, (3, 2, 4)), (1536, (128, 32, 32))])
def test_score_volume_matches_segment_volume_and_seg_stats(cuda_lib, C, shape):
    from cryovit_b200.host.metrics import SegStats

    D, h, w = shape
    head = _head(C, seed=C)
    g = torch.Generator().manual_seed(D)
    feats = torch.randn(C, D, h, w, generator=g).half().to(DEV)
    lab = _labels(D, 16 * h, 16 * w, seed=C + D)
    for thr in (0.5, 0.3):
        _, probs = head.segment_volume(feats, want_logits=False)
        ref = SegStats(probs, lab, thr).v
        got = head.score_volume(feats, lab, thr)
        assert got.dtype == torch.float64 and got.shape == (8,)
        assert torch.equal(got[COUNTS], ref[COUNTS]), (got.tolist(), ref.tolist())
        _close_soft(got, ref)
        # labels the fused path does not take (fp32) run segment_volume + seg_stats: the same numbers (seg_stats adds its
        # blocks with atomics, so the soft sums may differ in the last bits)
        fb = head.score_volume(feats, lab.float(), thr)
        assert torch.equal(fb[COUNTS], ref[COUNTS])
        _close_soft(fb, ref, 1e-12)
    if shape == (128, 32, 32):
        return
    head.rows8 = False  # CVIT_HEAD_ROWS8=0: the fallback on the other output-layer kernels
    _, probs = head.segment_volume(feats, want_logits=False)
    got, ref = head.score_volume(feats, lab), SegStats(probs, lab).v
    assert torch.equal(got[COUNTS], ref[COUNTS])
    _close_soft(got, ref, 1e-12)


# ----------------------------------------------------------------------------------------------- weight hand-over
@gpu
def test_head_refreshed_from_trainer_bucket_matches_load_state_dict(cuda_lib):
    from cryovit_b200.head import CryoVITHeadB200
    from cryovit_b200.train import CryoVITHeadTrainerB200
    from oracle import head as ohead

    C = 384
    tr = CryoVITHeadTrainerB200(C, lr=2e-3, state_dict=ohead.random_state_dict(C, seed=7))
    head = CryoVITHeadB200(C).cuda().attach_bucket(*tr.parameter_bucket())
    g = torch.Generator().manual_seed(1)
    feats = torch.randn(C, 3, 4, 5, generator=g).half().to(DEV)
    crop_f = torch.randn(C, 4, 3, 3, generator=g).half().to(DEV)
    crop_l = (torch.rand(4, 48, 48, generator=g) < 0.5).float().to(DEV)
    for steps in (0, 3):
        for _ in range(steps):
            tr.train_step(crop_f, crop_l)
        torch.cuda.synchronize()
        head.refresh()
        ref = CryoVITHeadB200(C).load_state_dict(tr.state_dict()).cuda()
        got_l, got_p = head.segment_volume(feats)
        ref_l, ref_p = ref.segment_volume(feats)
        assert torch.equal(got_l, ref_l) and torch.equal(got_p, ref_p), steps
        fe32 = feats.float()  # the bf16 projection (fp32 features) too
        assert torch.equal(head.segment_volume(fe32)[0], ref.segment_volume(fe32)[0])


# ----------------------------------------------------------------------------------------------- the loop
def _toy_split(root: Path, n_train: int, n_val: int, seed: int = 4):
    """Learnable toy tomograms (channel 0 carries the label), some voxels ignored; returns (train, val) TomoDatasets."""
    from cryovit.datasets import TomoDataset
    from cryovit_b200.host import hdf

    rng = np.random.default_rng(seed)
    recs = []
    for i in range(n_train + n_val):
        feats = (0.1 * rng.standard_normal((384, 4, 3, 3))).astype(np.float16)
        feats[0] = 2.0 * np.sign(rng.standard_normal((4, 3, 3)))
        lab = (np.repeat(np.repeat(feats[0].astype(np.float32), 16, axis=1), 16, axis=2) > 0).astype(np.int8)
        lab[0, :8] = -1
        hdf.write_tomogram(root / "S" / f"t{i}.hdf", {"data": np.zeros((4, 48, 48), np.uint8), "labels/mito": lab, "dino_features": feats})
        recs.append({"sample": "S", "tomo_name": f"t{i}.hdf"})
    mk = lambda r, train: TomoDataset(r, "dino_features", "mito", "split_id", root, train=train)
    return mk(recs[:n_train], True), mk(recs[n_train:], False), recs[n_train:]


def _validator(ds, **kw):
    from cryovit_b200.host.metrics import DiceLoss, DiceMetric, F1Metric
    from cryovit_b200.host.validate import Validator

    return Validator(ds, 384, {"dice_loss": DiceLoss()}, {"dice_metric": DiceMetric(0.5), "f1_metric": F1Metric()},
                     kw.get("every", 1), kw.get("limit", 1.0))


@gpu
def test_fit_head_validation_rows_match_the_metric_objects(cuda_lib, tmp_path):
    from cryovit_b200.head import CryoVITHeadB200
    from cryovit_b200.host import hdf
    from cryovit_b200.host.fit import fit_head
    from cryovit_b200.host.metrics import DiceLoss, DiceMetric, F1Metric
    from oracle import head as ohead

    train, val, val_recs = _toy_split(tmp_path, 3, 2)
    sd0 = ohead.random_state_dict(384, seed=5)
    hist = []
    sd = fit_head(train, in_channels=384, max_epochs=4, lr=2e-3, swa_epoch_start=None, exp_dir=tmp_path / "exp", state_dict=sd0,
                  validator=_validator(val), val_history=hist)
    assert [r["epoch"] for r in hist] == [0, 1, 2, 3]
    assert list(hist[-1]) == ["epoch", "dice_loss", "dice_metric", "f1_metric", "tomograms", "seconds"] and hist[-1]["tomograms"] == 2
    lines = (tmp_path / "exp" / "validation.csv").read_text().splitlines()
    assert lines[0] == "epoch,dice_loss,dice_metric,f1_metric,tomograms,seconds" and len(lines) == 5
    # the last row, independently: the returned weights, segment_volume, the metric objects
    head = CryoVITHeadB200(384).load_state_dict(sd).cuda()
    dl, dm, f1 = [], DiceMetric(0.5), F1Metric()
    for r in val_recs:
        f = hdf.read_tomogram(tmp_path / "S" / r["tomo_name"])
        _, probs = head.segment_volume(torch.from_numpy(f["dino_features"]).cuda(), want_logits=False)
        lab = torch.from_numpy(f["labels/mito"]).float().cuda()
        dl.append(float(DiceLoss()(probs, lab)))
        dm.update(probs, lab)
        f1.update(probs, lab)
    want = {"dice_loss": float(np.mean(dl)), "dice_metric": float(dm.compute()), "f1_metric": float(f1.compute())}
    for k, v in want.items():
        assert abs(hist[-1][k] - v) <= 1e-6, (k, hist[-1][k], v)


@gpu
def test_validation_leaves_training_untouched(cuda_lib, tmp_path):
    """Validation inside fit_head leaves the trainer exactly as it found it -- master weights, gradient bucket, AdamW
    moments, step count -- and draws nothing from numpy's or torch's global generators (the crop draws of the next epoch
    come from numpy's), so the training run is the one without validation. (Two fit_head runs are not compared bit for bit:
    the training step's reductions use atomics, and two runs WITHOUT validation already differ in the last bits.)"""
    from cryovit_b200.host.fit import fit_head
    from cryovit_b200.host.validate import Validator
    from oracle import head as ohead

    train, val, _ = _toy_split(tmp_path, 3, 2)
    base = _validator(val)
    checked = []

    class Watch(Validator):
        def run(self, trainer, epoch, cache_budget=0):
            state = [t.clone() for t in (trainer._flat_store, trainer.flat_g, trainer.flat_m, trainer.flat_v)]
            steps = trainer.step_count
            rng = (np.random.get_state(), torch.get_rng_state(), torch.cuda.get_rng_state())
            row = super().run(trainer, epoch, cache_budget)
            torch.cuda.synchronize()
            assert all(torch.equal(a, b) for a, b in zip(state, (trainer._flat_store, trainer.flat_g, trainer.flat_m, trainer.flat_v)))
            assert trainer.step_count == steps
            assert all(np.array_equal(a, b) for a, b in zip(rng[0], np.random.get_state()))
            assert torch.equal(rng[1], torch.get_rng_state()) and torch.equal(rng[2], torch.cuda.get_rng_state())
            checked.append(epoch)
            return row

    v = Watch(val, 384, base.losses, base.metrics, 1, 1.0)
    fit_head(train, in_channels=384, max_epochs=4, lr=2e-3, swa_epoch_start=2, state_dict=ohead.random_state_dict(384, seed=5), validator=v)
    assert checked == [0, 1, 2, 3]


@gpu
def test_rank_with_an_empty_shard_still_finishes(cuda_lib, tmp_path, monkeypatch):
    from cryovit_b200.train import CryoVITHeadTrainerB200
    from oracle import head as ohead

    _, val, _ = _toy_split(tmp_path, 0, 1)
    tr = CryoVITHeadTrainerB200(384, state_dict=ohead.random_state_dict(384, seed=5))
    monkeypatch.setenv("RANK", "1")
    monkeypatch.setenv("WORLD_SIZE", "2")  # no process group: the reduction is this rank's own (nothing)
    row = _validator(val).run(tr, 0)
    assert row["tomograms"] == 0 and row["dice_loss"] == 0.0 and row["dice_metric"] == 0.0


def _entry_data(tmp_path, n_per_sample=6):
    import pandas as pd
    from cryovit_b200.host import hdf

    rng = np.random.default_rng(4)
    rows = []
    for s in ("A", "B"):
        for i in range(n_per_sample):
            feats = (0.1 * rng.standard_normal((384, 4, 3, 3))).astype(np.float16)
            feats[0] = 2.0 * np.sign(rng.standard_normal((4, 3, 3)))
            lab = (np.repeat(np.repeat(feats[0].astype(np.float32), 16, axis=1), 16, axis=2) > 0).astype(np.int8)
            lab[0, :8] = -1
            hdf.write_tomogram(tmp_path / "data" / "tomograms" / s / f"{s}{i}.hdf",
                               {"data": rng.integers(0, 256, (4, 48, 48), dtype=np.uint8), "labels/mito": lab, "dino_features": feats})
            rows.append((s, f"{s}{i}.hdf", i % 2))
    (tmp_path / "data" / "csv").mkdir(parents=True, exist_ok=True)
    pd.DataFrame(rows, columns=["sample", "tomo_name", "split_id"]).to_csv(tmp_path / "data" / "csv" / "splits.csv", index=False)
    return ["model=cryovit", "+experiments=multi_mito", "datamodule.sample=[A,B]", "datamodule.split_id=0", "+model.in_channels=384",
            f"paths.data_dir={tmp_path / 'data'}"]


@gpu
def test_train_model_writes_validation_csv_on_the_lightning_schedule(cuda_lib, tmp_path):
    import pandas as pd
    from cryovit.config import compose
    from cryovit.run import train_model

    common = _entry_data(tmp_path)

    def run(tag, *extra):
        cfg = compose("train_model", common + [f"paths.exp_dir={tmp_path / tag}", "trainer.max_epochs=60", "model.lr=4e-4", *extra])
        w = train_model.run_trainer(cfg)
        return w, w.parent / "validation.csv"

    w_on, csv_on = run("on")
    df = pd.read_csv(csv_on)
    assert list(df.columns) == ["epoch", "dice_loss", "dice_metric", "f1_metric", "tomograms", "seconds"]
    assert df["epoch"].tolist() == list(range(60)) and (df["tomograms"] == 6).all()
    print(f"\n[validation] dice_metric epoch 0 {df['dice_metric'].iloc[0]:.3f} -> epoch 59 {df['dice_metric'].iloc[-1]:.3f}")
    assert df["dice_metric"].iloc[-1] > df["dice_metric"].iloc[0]
    _, csv3 = run("every3", "trainer.check_val_every_n_epoch=3")
    assert pd.read_csv(csv3)["epoch"].tolist() == list(range(2, 60, 3))
    w_off, csv_off = run("off", "trainer.limit_val_batches=0")  # validation off: no file, the weights as ever
    assert w_off.exists() and not csv_off.exists()


@gpu
def test_two_gpu_validation_with_an_empty_shard(cuda_lib, tmp_path):
    """torchrun with two ranks and ONE validation tomogram: rank 1 scores nothing but joins the reduction."""
    import pandas as pd
    from cryovit_b200.host import hdf

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    common = _entry_data(tmp_path, n_per_sample=3)
    df = pd.read_csv(tmp_path / "data" / "csv" / "splits.csv")
    keep = (df["split_id"] == 1) | (df["tomo_name"] == "A0.hdf")  # split 0 = one tomogram
    df[keep].to_csv(tmp_path / "data" / "csv" / "splits.csv", index=False)
    launch = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
              "--master-port", str(29300 + os.getpid() % 300)]
    env = dict(os.environ, PYTHONPATH=str(ROOT) + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run(launch + ["-m", "cryovit.training.train_model", *common, f"paths.exp_dir={tmp_path / 'exp'}",
                                 "trainer.max_epochs=3"], cwd=str(ROOT), env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    val = pd.read_csv(tmp_path / "exp" / "multi_cryovit_mito" / "A_B" / "split_0" / "validation.csv")
    assert val["epoch"].tolist() == [0, 1, 2] and (val["tomograms"] == 1).all()
