"""``cryovit.run.train_model`` for the CryoVIT head (reference run/train_model.py:156-312): experiment directory
layout, split-file data module, training with the reference's schedule, ``weights.pt`` with the reference's parameter
names. Lightning's ``Trainer`` is replaced by :func:`cryovit_b200.host.fit.fit_head` (native forward / backward /
NCCL all-reduce / AdamW step); W&B logging, ``torch.compile`` and checkpoint resume are not part of the hot path."""
from __future__ import annotations

import logging
from collections.abc import Iterable
from pathlib import Path

import torch

from .._lib import CryovitB200Error
from .config import instantiate
from .fit import fit_head
from .shard import process_group
from .validate import Validator


def _joined(x):
    return "_".join(sorted(x)) if not isinstance(x, str) and isinstance(x, Iterable) else x


def setup_exp_dir(cfg, create: bool = True):
    """train_model.py:156-203 / eval_model.py:103-141: ``exp_dir/<name>/<samples>[/split_<id>][/test_<samples>]``."""
    for k in ("model_dir", "data_dir", "exp_dir", "results_dir"):
        cfg.paths[k] = Path(cfg.paths[k])
    sample, test_sample = _joined(cfg.datamodule.sample), _joined(cfg.datamodule.get("test_sample"))
    new = cfg.paths.exp_dir / cfg.name / sample
    if cfg.datamodule.get("split_id") is not None:
        new = new / f"split_{cfg.datamodule.split_id}"
    if "Fractional" in cfg.datamodule["_target_"] and test_sample is not None:
        new = new / f"test_{test_sample}"
    if create:
        new.mkdir(parents=True, exist_ok=True)
    cfg.paths.exp_dir = new
    return cfg


def build_datamodule(cfg):
    """train_model.py:229-238: dataset / dataloader partials + the datamodule node's own keys."""
    node = {k: v for k, v in cfg.datamodule.items() if k not in ("dataset", "dataloader")}
    dataset_fn = instantiate(cfg.datamodule.dataset)
    split_file = Path(cfg.paths.data_dir) / cfg.paths.csv_name / cfg.paths.split_name
    return instantiate(node, split_file=split_file, dataset_fn=dataset_fn, dataloader_fn=None)


def build_validator(cfg, datamodule, in_channels: int) -> Validator | None:
    """Lightning's ``fit`` validates after every epoch by default: the datamodule's ``val_df()`` scored whole
    (``train=False``) with ``cfg.model``'s losses and metrics, on the schedule of ``trainer.check_val_every_n_epoch``
    and ``trainer.limit_val_batches``. None when that schedule validates nothing or the validation split is empty."""
    tr = cfg.trainer
    records = datamodule.val_df()
    if records.empty:
        logging.info("No validation data in the split file: training without validation.")
        return None
    losses = {k: instantiate(v) for k, v in (cfg.model.get("losses") or {}).items()}
    metrics = {k: instantiate(v) for k, v in (cfg.model.get("metrics") or {}).items()}
    v = Validator(datamodule.dataset_fn(records, train=False), in_channels, losses, metrics,
                  tr.get("check_val_every_n_epoch", 1), tr.get("limit_val_batches", 1.0))
    if v.count == 0:
        logging.info("trainer.limit_val_batches=%s: training without validation.", tr.get("limit_val_batches"))
        return None
    return v


def run_trainer(cfg) -> Path:
    """train_model.py:206-312. Returns the path of the saved ``weights.pt``. Under torchrun every rank binds its own
    GPU and joins one NCCL group for the gradient all-reduce (Lightning's DDP strategy in the reference)."""
    if cfg.model["_target_"] != "cryovit.models.CryoVIT":
        raise CryovitB200Error(f"model {cfg.model['_target_']} is outside the B200 hot path (CryoVIT head only)")
    with process_group():
        return _run_trainer(cfg)


def _run_trainer(cfg) -> Path:
    torch.manual_seed(cfg.random_seed)
    cfg = setup_exp_dir(cfg)
    datamodule = build_datamodule(cfg)
    logging.info("Setup dataset.")
    records = datamodule.train_df()
    if records.empty:
        raise ValueError("No training data found in the provided split file.")
    dataset = datamodule.dataset_fn(records, train=True)
    swa = cfg.get("callbacks", {}).get("stochastic_weight_average")
    max_epochs = int(cfg.trainer.max_epochs)
    swa_start = None
    if swa is not None:  # Lightning: a float swa_epoch_start is a fraction of max_epochs
        s = swa.get("swa_epoch_start", 0.8)
        swa_start = int(s * max_epochs) if isinstance(s, float) else int(s)
    ckpt = cfg.get("ckpt_path")
    state = None
    if ckpt:  # fine-tune from a .pt state dict or a .model file (run/train_model.py:118-137)
        if str(ckpt).endswith(".model"):
            from .model_io import load_model

            state = load_model(ckpt)[0].state_dict()
        elif str(ckpt).endswith(".pt"):
            state = torch.load(ckpt)
        else:
            raise ValueError(f"Unsupported checkpoint format: {Path(ckpt).suffix}. Use .pt or .model files.")
    in_channels = int(cfg.model.get("in_channels", 1536))
    validator = build_validator(cfg, datamodule, in_channels)
    logging.info("Starting training.")
    fit_head(dataset, in_channels=in_channels, max_epochs=max_epochs, lr=float(cfg.model.lr),
             weight_decay=float(cfg.model.get("weight_decay", 1e-3)), swa_epoch_start=swa_start, seed=int(cfg.random_seed),
             exp_dir=cfg.paths.exp_dir, state_dict=state, validator=validator)
    logging.info("Saving model.")
    return cfg.paths.exp_dir / "weights.pt"
