"""``datamodule.dataloader.batch_size`` in head training, without a GPU: the fit loop's batches (with a stub trainer), the
steps per epoch on one and on two ranks (gloo), the entry point's plumbing, and the refusals."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
DEPTHS = [3, 6, 4, 7, 5]  # an odd number of tomograms, all of different depths


def _tomos(root: Path, depths, planes=None):
    from cryovit_b200.host import hdf

    rng = np.random.default_rng(1)
    recs = []
    for i, d in enumerate(depths):
        h, w = planes[i] if planes else (33, 35)
        feats = rng.standard_normal((4, d, h, w)).astype(np.float16)
        lab = rng.integers(-1, 2, (d, 16 * h, 16 * w)).astype(np.int8)
        hdf.write_tomogram(root / "S" / f"t{i}.hdf", {"labels/mito": lab, "dino_features": feats})
        recs.append({"sample": "S", "tomo_name": f"t{i}.hdf"})
    return recs


class StubTrainer:
    """Records the steps it is given: ("step", features, labels) or ("batch", [(features, labels), ...])."""

    device = torch.device("cpu")
    seen: list = []

    def __init__(self, in_channels, lr, weight_decay, state_dict, seed):
        self.flat_p = torch.zeros(2)
        type(self).seen = []

    def sample_bytes(self, D, h, w):
        return 0

    def train_step(self, features, labels):
        type(self).seen.append(("step", [(features.clone(), labels.clone())]))
        self.flat_p += 1.0
        return torch.tensor(0.5)

    def train_batch(self, crops):
        type(self).seen.append(("batch", [(f.clone(), l.clone()) for f, l in crops]))
        self.flat_p += 1.0
        return torch.tensor(0.5)

    def state_dict(self):
        return {"w": self.flat_p.clone()}


def _plain_crops(ds, epochs: int, seed: int = 42) -> list:
    """What the plain ``dataset[i]`` loop draws, epoch by epoch: same order generator, same global crop generator."""
    np.random.seed(seed)
    order_rng, out = np.random.default_rng(seed), []
    for _ in range(epochs):
        out.append([(it.data, it.label) for it in (ds[int(i)] for i in order_rng.permutation(len(ds)))])
    return out


@pytest.mark.parametrize("batch_size", [2, 3])
@pytest.mark.parametrize("cache_gb", [1.0, 0.0])
def test_batches_are_the_consecutive_crops_of_the_plain_loop(tmp_path, monkeypatch, batch_size, cache_gb):
    from cryovit.datasets import TomoDataset
    from cryovit_b200.host import fit

    monkeypatch.setattr(fit, "CryoVITHeadTrainerB200", StubTrainer)
    ds = TomoDataset(_tomos(tmp_path, DEPTHS), "dino_features", "mito", "split_id", tmp_path, train=True)
    epochs = 3
    want = _plain_crops(ds, epochs)
    sd = fit.fit_head(ds, in_channels=4, max_epochs=epochs, swa_epoch_start=None, seed=42, cache_gb=cache_gb, batch_size=batch_size)
    got = StubTrainer.seen
    per_epoch = -(-len(DEPTHS) // batch_size)
    assert len(got) == epochs * per_epoch and torch.equal(sd["w"], torch.full((2,), float(epochs * per_epoch)))
    for e in range(epochs):
        steps = got[e * per_epoch:(e + 1) * per_epoch]
        assert all(kind == "batch" for kind, _ in steps)
        sizes = [len(crops) for _, crops in steps]
        assert sizes == [batch_size] * (per_epoch - 1) + [len(DEPTHS) - batch_size * (per_epoch - 1)]
        assert sizes[-1] < batch_size  # 5 crops divide by neither 2 nor 3: the last batch is the shorter one
        flat = [c for _, crops in steps for c in crops]
        assert len(flat) == len(want[e])
        for (f, l), (wf, wl) in zip(flat, want[e]):
            assert torch.equal(f, wf) and torch.equal(l, wl)
        assert len({c[0].shape[1] for c in flat}) > 1  # crops of different depths share batches


def test_batch_size_one_keeps_the_single_crop_step(tmp_path, monkeypatch):
    from cryovit.datasets import TomoDataset
    from cryovit_b200.host import fit

    monkeypatch.setattr(fit, "CryoVITHeadTrainerB200", StubTrainer)
    ds = TomoDataset(_tomos(tmp_path, DEPTHS), "dino_features", "mito", "split_id", tmp_path, train=True)
    want = _plain_crops(ds, 2)
    fit.fit_head(ds, in_channels=4, max_epochs=2, swa_epoch_start=None, seed=42, cache_gb=1.0)
    got = StubTrainer.seen
    assert [k for k, _ in got] == ["step"] * 2 * len(DEPTHS)
    assert all(torch.equal(c[0][0], w[0]) and torch.equal(c[0][1], w[1]) for (_, c), w in zip(got, want[0] + want[1]))


@pytest.mark.parametrize("bad", [0, -1, None, 2.0, True])
def test_fit_head_refuses_a_batch_size_that_is_not_a_positive_int(bad):
    from cryovit_b200.host.fit import fit_head

    with pytest.raises(ValueError, match="datamodule.dataloader.batch_size"):
        fit_head([], in_channels=4, batch_size=bad)


def test_fit_loop_refuses_a_batch_of_different_feature_planes(tmp_path, monkeypatch):
    """A 20x20 plane is not cropped (smaller than 32x32), a 33x35 one is cut to 32x32: the two cannot share a batch."""
    from cryovit.datasets import TomoDataset
    from cryovit_b200.host import fit

    monkeypatch.setattr(fit, "CryoVITHeadTrainerB200", StubTrainer)
    ds = TomoDataset(_tomos(tmp_path, [3, 4], planes=[(20, 20), (33, 35)]), "dino_features", "mito", "split_id", tmp_path, train=True)
    with pytest.raises(ValueError, match=r"different feature planes: S/t\d.hdf .* and S/t\d.hdf"):
        fit.fit_head(ds, in_channels=4, max_epochs=1, swa_epoch_start=None, seed=42, cache_gb=0.0, batch_size=2)
    assert StubTrainer.seen == []  # refused before the step


def test_cache_budget_sets_aside_the_batch(monkeypatch):
    from cryovit_b200.host import fit

    monkeypatch.delenv("CRYOVIT_B200_FEATURE_CACHE_GB", raising=False)
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda: (100_000, 200_000))
    assert fit._cache_budget_bytes(None) == 60_000
    assert fit._cache_budget_bytes(None, reserve=50_000) == 30_000
    assert fit._cache_budget_bytes(None, reserve=500_000) == 0
    assert fit._cache_budget_bytes(2.0, reserve=50_000) == 2_000_000_000  # an explicit budget is the user's


# ----------------------------------------------------------------------------------------------- two ranks (gloo)
WORKER = r'''
import os, sys
from pathlib import Path
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["REPO"])
sys.path.insert(0, os.environ["TESTS"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + os.environ["PORT"], rank=int(os.environ["RANK"]),
                        world_size=int(os.environ["WORLD_SIZE"]))
from cryovit.datasets import TomoDataset
from cryovit_b200.host import fit
from test_train_batch_host import StubTrainer
fit.CryoVITHeadTrainerB200 = StubTrainer
root = Path(os.environ["WORK"])
recs = [{"sample": "S", "tomo_name": f"t{i}.hdf"} for i in range(int(os.environ["N"]))]
ds = TomoDataset(recs, "dino_features", "mito", "split_id", root, train=True)
fit.fit_head(ds, in_channels=4, max_epochs=2, swa_epoch_start=None, seed=42, cache_gb=0.0, batch_size=int(os.environ["B"]))
sizes = [len(c) for _, c in StubTrainer.seen]
(root / f"steps_{dist.get_rank()}.txt").write_text(" ".join(map(str, sizes)))
dist.barrier()
dist.destroy_process_group()
'''


def test_two_ranks_take_the_same_number_of_steps(tmp_path):
    """7 tomograms on 2 ranks: 6 usable, a share of 3 per rank, batches of 2 -> steps of 2 and 1 crops on both ranks."""
    n, b = 7, 2
    _tomos(tmp_path, [3, 6, 4, 7, 5, 3, 4])
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    port = str(31500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", PORT=port, WORK=str(tmp_path), REPO=str(ROOT), TESTS=str(ROOT / "tests"),
                   N=str(n), B=str(b), CUDA_VISIBLE_DEVICES="")
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=240)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(outs)
    steps = [(tmp_path / f"steps_{r}.txt").read_text().split() for r in range(2)]
    assert steps[0] == steps[1] == ["2", "1", "2", "1"]  # two epochs of (2, 1)


# ----------------------------------------------------------------------------------------------- entry point plumbing
def _entry_data(tmp_path):
    import pandas as pd
    from cryovit_b200.host import hdf

    rng = np.random.default_rng(4)
    rows = []
    for s in ("A", "B"):
        for i in range(4):
            feats = (0.1 * rng.standard_normal((384, 4, 3, 3))).astype(np.float16)
            lab = (rng.random((4, 48, 48)) < 0.3).astype(np.int8)
            hdf.write_tomogram(tmp_path / "data" / "tomograms" / s / f"{s}{i}.hdf",
                               {"data": rng.integers(0, 256, (4, 48, 48), dtype=np.uint8), "labels/mito": lab, "dino_features": feats})
            rows.append((s, f"{s}{i}.hdf", i % 2))
    (tmp_path / "data" / "csv").mkdir(parents=True, exist_ok=True)
    pd.DataFrame(rows, columns=["sample", "tomo_name", "split_id"]).to_csv(tmp_path / "data" / "csv" / "splits.csv", index=False)
    return ["model=cryovit", "+experiments=multi_mito", "datamodule.sample=[A,B]", "datamodule.split_id=0", "+model.in_channels=384",
            f"paths.data_dir={tmp_path / 'data'}", f"paths.exp_dir={tmp_path / 'exp'}"]


@pytest.mark.parametrize("override, want", [(None, 1), ("datamodule.dataloader.batch_size=1", 1),
                                            ("datamodule.dataloader.batch_size=2", 2), ("datamodule.dataloader.batch_size=4", 4)])
def test_run_trainer_passes_the_dataloader_batch_size_to_fit_head(tmp_path, monkeypatch, override, want):
    from cryovit.config import compose
    from cryovit_b200.host import train_model

    got = {}
    monkeypatch.setattr(train_model, "fit_head", lambda *a, **kw: got.update(kw) or {})
    cfg = compose("train_model", _entry_data(tmp_path) + ([override] if override else []))
    train_model.run_trainer(cfg)
    assert got["batch_size"] == want and type(got["batch_size"]) is int


@pytest.mark.parametrize("bad", ["0", "-1", "null"])
def test_run_trainer_refuses_a_bad_dataloader_batch_size(tmp_path, monkeypatch, bad):
    from cryovit.config import compose
    from cryovit_b200.host import train_model

    monkeypatch.setattr(train_model, "fit_head", lambda *a, **k: pytest.fail("fit_head reached"))
    cfg = compose("train_model", _entry_data(tmp_path) + [f"datamodule.dataloader.batch_size={bad}"])
    with pytest.raises(ValueError, match="datamodule.dataloader.batch_size"):
        train_model.run_trainer(cfg)
