"""CPU suite for the host-side mirror of the reference interfaces (cryovit_b200/host, re-exported as ``cryovit.*``):
config composition, the tomogram file layout, crop / collate against golden vectors produced by the reference's own
source (tests/golden/reference_src.npz), sharding, and a world_size-2 gloo run of the multi-rank paths."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
GOLD = ROOT / "tests" / "golden"


@pytest.fixture(scope="module")
def ref():
    return np.load(GOLD / "reference_src.npz")


# ------------------------------------------------------------------------------------------------- config (seam B1)
def test_compose_dino_features_defaults_and_overrides():
    from cryovit.config import compose, missing_keys

    cfg = compose("dino_features", ["sample=Q18", "paths.data_dir=/data/x", "batch_size=64", "paths=default"])
    assert cfg.batch_size == 64 and cfg.sample == "Q18" and cfg.export_features is False and cfg.use_sam is False
    assert cfg.paths.data_dir == "/data/x" and cfg.paths.tomo_name == "tomograms" and cfg.paths.feature_name == "dino_features"
    assert cfg.paths.results_dir == cfg.paths.exp_dir  # ${paths.exp_dir}
    assert cfg.model_dir == f"{cfg.paths.model_dir}/DINOv2"  # ${paths.model_dir}/${paths.dino_name}
    ds, dl = cfg.datamodule.dataset, cfg.datamodule.dataloader
    assert ds["_target_"] == "cryovit.datasets.VITDataset" and ds["_partial_"] is True
    assert ds["data_root"] == "/data/x/tomograms"
    # datamodule/dino.yaml overrides the loader defaults: one whole tomogram per item, no workers
    assert dl["batch_size"] is None and dl["num_workers"] == 0 and dl["pin_memory"] is True
    assert missing_keys(cfg) == []


def test_missing_mandatory_keys_exit(tmp_path, caplog):
    from cryovit.config import compose, validate_dino_config

    (tmp_path / "paths").mkdir()
    (tmp_path / "paths" / "default.yaml").write_text("model_dir: ???\ndata_dir: /d\nexp_dir: /e\nresults_dir: /r\n")
    (tmp_path / "dino_features.yaml").write_text("defaults:\n  - paths: default\n  - _self_\nmodel_dir: /m\nsample: null\ndatamodule: {}\n")
    cfg = compose("dino_features", [], config_dir=tmp_path)
    with pytest.raises(SystemExit) as e:
        validate_dino_config(cfg)
    assert e.value.code == 1  # config.py:227-229


def test_model_config_targets_resolve():
    from cryovit.config import compose, instantiate

    cfg = compose("model/cryovit", [])
    assert cfg["_target_"] == "cryovit.models.CryoVIT" and cfg["input_key"] == "dino_features" and cfg["lr"] == 1e-4
    assert set(cfg["losses"]) == {"dice_loss"} and set(cfg["metrics"]) == {"dice_metric", "f1_metric"}
    m = instantiate(cfg["metrics"]["dice_metric"])
    assert m.threshold == 0.5


# ------------------------------------------------------------------------------------------------- file layout (B5)
def test_save_data_layout_roundtrip(tmp_path):
    from cryovit.run.dino_features import _save_data
    from cryovit_b200.host import hdf

    rng = np.random.default_rng(0)
    src = {"data": rng.integers(0, 256, (4, 32, 48), dtype=np.uint8), "mito": rng.integers(-1, 2, (4, 32, 48)).astype(np.int8),
           "granule": rng.integers(-1, 2, (4, 32, 48)).astype(np.int8), "dino_features": np.zeros((2, 4, 2, 3), np.float16)}
    feats = rng.standard_normal((384, 4, 2, 3)).astype(np.float16)
    _save_data(src, feats, "t0.hdf", tmp_path / "out" / "S")
    path = tmp_path / "out" / "S" / "t0.hdf"
    assert sorted(hdf.list_keys(path)) == ["data", "dino_features", "labels/granule", "labels/mito"]
    back = hdf.read_tomogram(path)
    assert back["dino_features"].dtype == np.float16 and back["dino_features"].shape == (384, 4, 2, 3)
    assert np.array_equal(back["dino_features"], feats)  # the stale source features were replaced
    assert np.array_equal(back["data"], src["data"]) and back["data"].dtype == np.uint8
    assert np.array_equal(back["labels/mito"], src["mito"]) and back["labels/mito"].dtype == np.int8
    _save_data({"data": src["data"]}, feats[:1], "t0.hdf", tmp_path / "out" / "S")  # "w": overwrite, no merge
    assert sorted(hdf.list_keys(path)) == ["data", "dino_features"]
    # SURVEY 8f row f2's option: the features in depth slabs (the default above is the reference's contiguous layout)
    _save_data({"data": src["data"]}, feats, "t1.hdf", tmp_path / "out" / "S", feature_chunk_depth=3)
    assert np.array_equal(hdf.read_tomogram(tmp_path / "out" / "S" / "t1.hdf", keys=["dino_features"])["dino_features"], feats)
    if hdf.backend() == "hdf5-classic":
        from cryovit_b200.host import hdf5_classic

        with hdf5_classic.File(tmp_path / "out" / "S" / "t1.hdf") as fh:
            assert fh.info("dino_features").chunks == (384, 3, 2, 3) and fh.info("dino_features").filters == []
        with hdf5_classic.File(path) as fh:
            assert fh.info("dino_features").layout == "contiguous" and fh.info("data").layout == "chunked"


# ------------------------------------------------------------------------------------------------- crop / collate (a8)
def test_random_crop_matches_reference(ref):
    from cryovit.datasets import TomoDataset

    ds = TomoDataset([], "dino_features", "mito", "split_id", Path("."), train=True)
    rng = np.random.default_rng(5)
    feat = rng.standard_normal((6, 140, 34, 33)).astype(np.float16)
    label = rng.integers(-1, 2, size=(140, 34 * 16, 33 * 16)).astype(np.int8)
    rec = {"input": feat, "label": label}
    np.random.seed(123)
    ds._random_crop(rec)
    assert tuple(rec["input"].shape) == tuple(ref["crop_input_shape"]) == (6, 128, 32, 32)
    assert tuple(rec["label"].shape) == tuple(ref["crop_label_shape"]) == (128, 512, 512)
    assert rec["input"].astype(np.float64).sum() == float(ref["crop_input_sum"])
    assert rec["label"].astype(np.int64).sum() == int(ref["crop_label_sum"])


def test_collate_matches_reference_and_pads_ragged(ref):
    from cryovit.datamodules.utils import collate_fn
    from cryovit.types import TomogramData

    items = [TomogramData("S", f"t{i}", i, torch.from_numpy(ref["collate_in_data"][i]), torch.from_numpy(ref["collate_in_label"][i]), {})
             for i in range(2)]
    b = collate_fn(items)
    assert b.tomo_batch.dtype == torch.float32 and tuple(b.tomo_batch.shape) == (2, 4, 6, 3, 2)
    assert np.array_equal(b.tomo_batch.numpy(), ref["collate_tomo_batch"])
    assert np.array_equal(b.labels.numpy(), ref["collate_labels"])
    assert np.array_equal(b.tomo_sizes.numpy(), ref["collate_tomo_sizes"])
    assert b.metadata.identifiers() == (["S", "S"], ["t0", "t1"]) and b.metadata.split_id.tolist() == [0, 1]
    # ragged depths: data padded with 0, labels with -1 (ignored by the masked loss)
    short = TomogramData("S", "t2", 2, items[0].data[:, :3], items[0].label[:3], {})
    b2 = collate_fn([items[0], short])
    assert b2.tomo_sizes.tolist() == [4, 3] and b2.min_slices == 3
    assert torch.all(b2.labels[1, 3] == -1) and torch.all(b2.tomo_batch[1, 3] == 0)


def test_tomo_dataset_reads_layout(tmp_path):
    from cryovit.datasets import TomoDataset
    from cryovit_b200.host import hdf

    rng = np.random.default_rng(1)
    feats = rng.standard_normal((8, 5, 2, 2)).astype(np.float16)
    lab = rng.integers(-1, 2, (5, 32, 32)).astype(np.int8)
    hdf.write_tomogram(tmp_path / "S" / "a.hdf", {"data": np.zeros((5, 32, 32), np.uint8), "labels/mito": lab, "dino_features": feats})
    ds = TomoDataset([{"sample": "S", "tomo_name": "a.hdf", "split_id": 3}], "dino_features", "mito", "split_id", tmp_path)
    it = ds[0]
    assert it.split_id == 3 and tuple(it.data.shape) == (8, 5, 2, 2) and it.data.dtype == torch.float16
    assert np.array_equal(it.label.numpy(), lab)
    with pytest.raises(IndexError):
        ds[1]


# ------------------------------------------------------------------------------------------------- sharding (8e)
@pytest.mark.parametrize("n,world", [(128, 8), (128, 3), (5, 8), (0, 2), (1029, 4)])
def test_shard_range_partitions(n, world):
    from cryovit_b200.host.shard import shard_range, shard_round_robin

    parts = [shard_range(n, r, world) for r in range(world)]
    assert [i for p in parts for i in p] == list(range(n))  # contiguous, ordered, complete, disjoint
    assert max(len(p) for p in parts) - min(len(p) for p in parts) <= 1
    rr = [shard_round_robin(list(range(n)), r, world) for r in range(world)]
    assert sorted(i for p in rr for i in p) == list(range(n))


WORKER = r'''
import os, sys
from pathlib import Path
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["REPO"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + os.environ["PORT"], rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
from cryovit_b200.host import dino_features as df, hdf
from cryovit_b200.host.metrics import _MeanOfBatchesMetric
from cryovit.config import compose
rank = dist.get_rank()
# (1) tomograms of a sample are dealt round-robin; every rank writes only its own files (stub extractor: no GPU here)
df._dino_features = lambda data, model, bs: np.full((4, data.shape[0], 2, 3), float(data.float().mean()), np.float16)
root = Path(os.environ["WORK"])
cfg = compose("dino_features", [f"paths.data_dir={root}", f"paths.exp_dir={root}/exp", "sample=Q18"])
done = df._process_sample(root / "dino_features", root / "tomograms", root / "csv", None, "Q18", cfg["datamodule"], 2)
(root / f"done_{rank}.txt").write_text("\n".join(done))
# (2) metric states reduce with "sum" across ranks (metrics.py:24-27 semantics)
m = _MeanOfBatchesMetric()
m._add(torch.tensor(0.25 if rank == 0 else 0.75, dtype=torch.float64))
if rank == 1:
    m._add(torch.tensor(0.5, dtype=torch.float64))
m.all_reduce()
assert abs(float(m.compute()) - 0.5) < 1e-12 and m.total == 3.0, (float(m.compute()), m.total)
# (3) head training: one flat gradient bucket, summed over ranks (the 1/world factor rides on the loss gradient)
from cryovit_b200.train import allreduce_gradient_bucket
bucket = torch.full((1000,), float(rank + 1)) / dist.get_world_size()
allreduce_gradient_bucket(bucket)
assert torch.allclose(bucket, torch.full((1000,), 1.5)), bucket[:4]
dist.barrier()
dist.destroy_process_group()
'''


def test_two_rank_gloo_sharded_extraction_and_metric_reduce(tmp_path):
    from cryovit_b200.host import hdf

    rng = np.random.default_rng(2)
    names = [f"tomo_{i}.hdf" for i in range(5)]
    for i, n in enumerate(names):
        hdf.write_tomogram(tmp_path / "dino_features" / "Q18" / n, {"data": rng.integers(0, 256, (3 + i, 32, 48), dtype=np.uint8),
                                                                    "labels/mito": np.zeros((3 + i, 32, 48), np.int8)})
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    port = str(29500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", PORT=port, WORK=str(tmp_path), REPO=str(ROOT))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=240)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(outs)
    done = [(tmp_path / f"done_{r}.txt").read_text().split() for r in range(2)]
    assert done[0] == names[0::2] and done[1] == names[1::2]  # disjoint, complete, no collective needed
    for i, n in enumerate(names):
        back = hdf.read_tomogram(tmp_path / "tomograms" / "Q18" / n)
        assert sorted(back) == ["data", "dino_features", "labels/mito"]
        assert back["dino_features"].shape == (4, 3 + i, 2, 3) and back["data"].shape == (3 + i, 32, 48)


PG_WORKER = r'''
import os, sys
import torch, torch.distributed as dist
sys.path.insert(0, os.environ["REPO"])
from cryovit_b200.host import shard
from cryovit_b200.host.eval_model import _merge_rows
rank, world = shard.rank_world()
assert world == 2 and not dist.is_initialized()
try:
    shard.require_process_group("fit_head")
    raise SystemExit("require_process_group accepted WORLD_SIZE=2 without a process group")
except RuntimeError as e:
    assert "WORLD_SIZE=2" in str(e)
from cryovit_b200.host import fit
try:  # the training loop refuses BEFORE it touches a device: no rank trains alone on a share of the data
    fit.fit_head([], in_channels=384)
    raise SystemExit("fit_head ran without a process group")
except RuntimeError as e:
    assert "not initialised" in str(e)
with shard.process_group(need_collectives=False):
    assert not dist.is_initialized()          # feature extraction: ranks only split an index range
with shard.process_group():                    # train / eval entry points: launcher env -> gloo here, NCCL on a GPU box
    assert dist.is_initialized() and dist.get_world_size() == 2 and dist.get_rank() == rank
    shard.require_process_group("fit_head")
    class W:
        rows = []
        def on_test_batch_end(self, res): self.rows.append(res)
    w = W()
    _merge_rows([f"row-of-rank-{rank}"], [w], rank, world)
    assert (w.rows == ["row-of-rank-0", "row-of-rank-1"]) if rank == 0 else (w.rows == [])
assert not dist.is_initialized()               # torn down again: it was created here
'''


def test_entry_point_process_group_plumbing_two_ranks(tmp_path):
    """ADVICE r1 (high): under torchrun the train / eval entry points must join ONE process group (gradient all-reduce,
    csv row gather) and bind their own GPU; a loop that shards by RANK without a group must refuse to run. Launched
    the way torchrun launches (RANK / LOCAL_RANK / WORLD_SIZE / MASTER_ADDR / MASTER_PORT): NCCL with one GPU per rank
    where there are two, gloo otherwise (NCCL refuses two ranks on one GPU, so the ranks are then shown no GPU)."""
    script = tmp_path / "pg_worker.py"
    script.write_text(PG_WORKER)
    port = str(31500 + os.getpid() % 2000)
    gpus = {} if torch.cuda.device_count() >= 2 else {"CUDA_VISIBLE_DEVICES": ""}
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), LOCAL_RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=port, REPO=str(ROOT),
                   **gpus)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=240)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(outs)


def test_wpack_weight_image_is_the_banded_matrix():
    """csrc/conv_wpack.cu's B operand: entry [kh][step][chunk][block][j_out][co][ci] is w[co, ci, kd = 2 - block, kh,
    kw = j_in - j_out] where j_in = 2 step + chunk, zero outside the three taps."""
    from cryovit_b200.head import wpack_weight_image

    for cout, P in ((8, 8), (1, 16)):
        w = torch.randn(cout, 8, 3, 3, 3, generator=torch.Generator().manual_seed(cout))
        img = wpack_weight_image(w, P).reshape(3, (P + 2) // 2, 2, 3, P, cout, 8)
        for kh, st, c, blk, jo in ((0, 0, 0, 0, 0), (1, 2, 1, 2, 3), (2, (P + 1) // 2, (P + 1) % 2, 1, P - 1), (1, 0, 1, 1, 5)):
            kw = 2 * st + c - jo
            want = w[:, :, 2 - blk, kh, kw] if 0 <= kw <= 2 else torch.zeros(cout, 8)
            assert torch.equal(img[kh, st, c, blk, jo], want), (cout, P, kh, st, c, blk, jo)
        assert int((img != 0).sum()) == 27 * cout * 8 * P  # every tap appears once per packed output voxel


def test_dino_features_argument_errors_match_the_reference():
    """Host-side argument handling of the extractor seam (run/dino_features.py:31-64), checked before any GPU work: an
    empty tomogram fails like the reference's ``np.concatenate([])``, a zero batch size like its ``range(0, D, 0)``,
    and shapes the 14-pixel patch grid cannot tile are refused."""
    import torch

    from cryovit_b200._lib import CryovitB200Error
    from cryovit_b200.extract import _dino_features
    from cryovit_b200.vit import build_model

    m = build_model("dinov2_vits14_reg")
    with pytest.raises(ValueError, match="at least one array"):
        _dino_features(torch.zeros(0, 3, 28, 28), m, 4)
    with pytest.raises(CryovitB200Error):
        _dino_features(torch.zeros(2, 3, 30, 28), m, 4)
    with pytest.raises(CryovitB200Error):
        _dino_features(torch.zeros(2, 1, 28, 28), m, 4)
    with pytest.raises(CryovitB200Error):
        _dino_features(torch.zeros(2, 3, 28, 28), object(), 4)


def test_operand_format_switch(monkeypatch):
    """The 16-bit format of the bounded ViT operands: constructor argument, CRYOVIT_B200_OPERANDS for the Hydra entry
    points, "mixed-attn" by default (fp16 norm1 / attention output and their weights, bf16 q/k/v, probabilities and FFN);
    anything else is refused before any GPU work."""
    import torch

    from cryovit_b200._lib import CryovitB200Error
    from cryovit_b200.vit import DinoVisionTransformerB200, build_model

    monkeypatch.delenv("CRYOVIT_B200_OPERANDS", raising=False)
    m = build_model("dinov2_vits14_reg")
    assert (m.operands, m.operand_dtype, m.qkv_dtype, m.ffn_dtype) == ("mixed-attn", torch.float16, torch.bfloat16, torch.bfloat16)
    m = build_model("dinov2_vits14_reg", operands="mixed")
    assert (m.operands, m.operand_dtype, m.qkv_dtype, m.ffn_dtype) == ("mixed", torch.float16, torch.bfloat16, torch.float16)
    m = build_model("dinov2_vits14_reg", operands=torch.float16)
    assert (m.operands, m.operand_dtype, m.qkv_dtype) == ("fp16", torch.float16, torch.float16)
    monkeypatch.setenv("CRYOVIT_B200_OPERANDS", "bf16")
    m = build_model("dinov2_vits14_reg")
    assert (m.operands, m.operand_dtype, m.qkv_dtype) == ("bf16", torch.bfloat16, torch.bfloat16)
    assert build_model("dinov2_vits14_reg", operands="fp16").operands == "fp16"  # argument wins
    monkeypatch.setenv("CRYOVIT_B200_OPERANDS", "fp8")
    with pytest.raises(CryovitB200Error):
        build_model("dinov2_vits14_reg")
    with pytest.raises(CryovitB200Error):
        DinoVisionTransformerB200("dinov2_vits14_reg", torch.float32)


def test_load_model_refuses_to_run_without_a_checkpoint(tmp_path):
    """run/dino_features.py:335-337: the reference fails when torch.hub cannot deliver the model; so does the mirror.
    Random weights need the explicit ``allow_random_weights`` override (checked before any GPU work)."""
    from cryovit_b200.host import dino_features as df

    with pytest.raises(FileNotFoundError, match="allow_random_weights"):
        df.load_model(tmp_path, "dinov2_vits14_reg")
    with pytest.raises(FileNotFoundError):
        df.load_model(None)
    assert "dinov2_vitg14_reg4_pretrain.pth" in df.checkpoint_names("dinov2_vitg14_reg")
    assert "dinov2_vits14_reg4_pretrain.pth" in df.checkpoint_names("dinov2_vits14_reg")


def test_process_sample_overlaps_io_and_can_resume(tmp_path, monkeypatch):
    """``_process_sample`` (run/dino_features.py:156-205) with the read of tomogram i+1 and the write of tomogram i-1
    overlapped with the extraction of tomogram i (stub extractor: no GPU here): same files, same keys and record order as
    the serial loop; the reader really runs ahead; an error in the writer thread surfaces in the call; ``skip_existing``
    resumes an interrupted run without touching finished files."""
    import threading

    from cryovit.config import compose
    from cryovit_b200.host import dino_features as df, hdf

    rng = np.random.default_rng(4)
    names = [f"tomo_{i}.hdf" for i in range(4)]
    for i, n in enumerate(names):
        hdf.write_tomogram(tmp_path / "dino_features" / "Q18" / n, {"data": rng.integers(0, 256, (2 + i, 32, 48), dtype=np.uint8),
                                                                    "labels/mito": np.full((2 + i, 32, 48), i, np.int8)})
    cfg = compose("dino_features", [f"paths.data_dir={tmp_path}", f"paths.exp_dir={tmp_path}/exp", "sample=Q18"])
    events, main_thread = [], threading.get_ident()
    real_read = df._read_source

    def spy_read(path):
        events.append(("read", Path(path).name, threading.get_ident() != main_thread))
        return real_read(path)

    def fake_features(data, model, bs):
        events.append(("extract", int(data.shape[0]), False))
        return np.full((4, data.shape[0], 2, 3), float(data.float().mean()), np.float16)

    monkeypatch.setattr(df, "_read_source", spy_read)
    monkeypatch.setattr(df, "_dino_features", fake_features)
    args = (tmp_path / "dino_features", tmp_path / "tomograms", tmp_path / "csv", None, "Q18", cfg["datamodule"], 2)
    assert df._process_sample(*args) == names
    assert all(off_main for kind, _, off_main in events if kind == "read"), "reads must run on the reader thread"
    # the read of tomogram 1 was submitted before tomogram 0 was extracted: it appears before the SECOND extract
    order = [(k, v) for k, v, _ in events]
    assert order.index(("read", names[1])) < order.index(("extract", 3))
    for i, n in enumerate(names):
        back = hdf.read_tomogram(tmp_path / "tomograms" / "Q18" / n)
        assert sorted(back) == ["data", "dino_features", "labels/mito"]
        assert back["dino_features"].shape == (4, 2 + i, 2, 3) and (back["labels/mito"] == i).all()
    # resume: nothing left to do, nothing read, nothing rewritten
    stamp = {n: (tmp_path / "tomograms" / "Q18" / n).stat().st_mtime_ns for n in names}
    events.clear()
    assert df._process_sample(*args, skip_existing=True) == []
    assert not events and stamp == {n: (tmp_path / "tomograms" / "Q18" / n).stat().st_mtime_ns for n in names}
    (tmp_path / "tomograms" / "Q18" / names[2]).unlink()
    assert df._process_sample(*args, skip_existing=True) == [names[2]]
    # a failing writer surfaces inside the call
    monkeypatch.setattr(df, "_save_data", lambda *a, **k: (_ for _ in ()).throw(OSError("disk full")))
    with pytest.raises(OSError, match="disk full"):
        df._process_sample(*args)


def test_resident_cache_gives_the_same_items_as_the_dataset(tmp_path):
    """ResidentTomoCache (the fit loop's HBM-resident training set; here on the CPU device): same records, same crop
    draws and same tensors as ``dataset[i]`` under the same seed, one file read per tomogram however many epochs, and
    items past the budget still served (from their file)."""
    from cryovit.datasets import TomoDataset
    from cryovit_b200.host import hdf
    from cryovit_b200.host.datasets import ResidentTomoCache

    rng = np.random.default_rng(0)
    recs = []
    for i, (d, h) in enumerate([(5, 34), (3, 32), (6, 40)]):
        feats = rng.standard_normal((8, d, h, 36)).astype(np.float16)
        lab = rng.integers(-1, 2, (d, 16 * h, 16 * 36)).astype(np.int8)
        hdf.write_tomogram(tmp_path / "S" / f"t{i}.hdf", {"data": np.zeros((d, 16, 16), np.uint8), "labels/mito": lab, "dino_features": feats})
        recs.append({"sample": "S", "tomo_name": f"t{i}.hdf", "split_id": i})
    order = [0, 1, 2, 2, 0, 1, 1, 0, 2]
    ds = TomoDataset(recs, "dino_features", "mito", "split_id", tmp_path, train=True)
    np.random.seed(7)
    plain = [ds[i] for i in order]
    first_item_bytes = 8 * 5 * 34 * 36 * 2 + 5 * (16 * 34) * (16 * 36)  # fp16 features + int8 labels of t0
    for budget, kept in ((1 << 30, 3), (first_item_bytes + 10, 1)):
        cache = ResidentTomoCache(ds, "cpu", budget)
        np.random.seed(7)
        got = [cache.get(i) for i in order]
        for a, b in zip(plain, got):
            assert (a.sample, a.tomo_name, a.split_id) == (b.sample, b.tomo_name, b.split_id)
            assert a.data.shape[-2:] == (32, 32) and torch.equal(a.data, b.data) and torch.equal(a.label, b.label)
            assert b.data.is_contiguous() and b.label.is_contiguous()
        assert len(cache._items) == kept
        assert cache.file_reads == (3 if kept == 3 else 1 + sum(1 for i in order if i != 0))


def test_fit_loop_schedule_cache_and_prefetch_with_a_stub_trainer(tmp_path, monkeypatch):
    """host/fit.py without a GPU: the trainer is a stub that records what it is given. The loop must (a) walk a fresh
    permutation of the dataset per epoch, (b) hand the trainer exactly the crops the plain ``dataset[i]`` loop draws under
    the same seed, with or without the resident cache, (c) read every tomogram file once when the cache holds the set
    and once per use when it is off, (d) average the weights of the epoch starts from ``swa_epoch_start`` on."""
    from cryovit.datasets import TomoDataset
    from cryovit_b200.host import fit, hdf

    rng = np.random.default_rng(1)
    recs = []
    for i in range(3):
        feats = rng.standard_normal((4, 3 + i, 33, 35)).astype(np.float16)
        lab = rng.integers(-1, 2, (3 + i, 16 * 33, 16 * 35)).astype(np.int8)
        hdf.write_tomogram(tmp_path / "S" / f"t{i}.hdf", {"labels/mito": lab, "dino_features": feats})
        recs.append({"sample": "S", "tomo_name": f"t{i}.hdf"})

    class StubTrainer:
        device = torch.device("cpu")
        seen: list = []

        def __init__(self, in_channels, lr, weight_decay, state_dict, seed):
            self.flat_p = torch.zeros(2)
            type(self).seen = []

        def train_step(self, features, labels):
            assert features.shape[-2:] == (32, 32) and labels.shape[-2:] == (512, 512) and features.is_contiguous()
            type(self).seen.append((features.clone(), labels.clone()))
            self.flat_p += 1.0  # "weights" = number of steps taken
            return torch.tensor(0.5)

        def state_dict(self):
            return {"w": self.flat_p.clone()}

    monkeypatch.setattr(fit, "CryoVITHeadTrainerB200", StubTrainer)
    reads = []
    real = hdf.read_tomogram
    monkeypatch.setattr(hdf, "read_tomogram", lambda path, keys=None: (reads.append(Path(path).name), real(path, keys))[1])
    epochs = 4
    ds = TomoDataset(recs, "dino_features", "mito", "split_id", tmp_path, train=True)
    # what the plain loop would feed: same order generator, same global crop generator
    np.random.seed(42)
    order_rng, want = np.random.default_rng(42), []
    for _ in range(epochs):
        for i in order_rng.permutation(3):
            it = ds[int(i)]
            want.append((it.data, it.label))
    for cache_gb, n_reads in ((1.0, 3), (0.0, 3 * epochs)):
        reads.clear()
        secs: list = []
        sd = fit.fit_head(ds, in_channels=4, max_epochs=epochs, swa_epoch_start=2, seed=42, cache_gb=cache_gb, epoch_seconds=secs)
        got = StubTrainer.seen
        assert len(got) == len(want) == 3 * epochs and len(secs) == epochs
        assert all(torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) for a, b in zip(got, want))
        assert len(reads) == n_reads and (cache_gb == 0.0 or sorted(reads) == ["t0.hdf", "t1.hdf", "t2.hdf"])
        # SWA: mean of the weights at the starts of epochs 2 and 3 = (6 + 9) / 2 steps
        assert torch.allclose(sd["w"], torch.full((2,), 7.5))
