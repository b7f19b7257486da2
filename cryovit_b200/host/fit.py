"""Head training loop with the reference's schedule (run/train_model.py:206-312, configs/trainer/fit.yaml,
configs/callbacks/stochastic_weight_average.yaml): seed, AdamW(lr, weight_decay) on every step, batch of ONE tomogram
crop per process (dataloader/default.yaml batch_size 1), ``max_epochs`` passes, stochastic weight averaging of the
weights from ``swa_epoch_start`` on (constant learning rate ``swa_lrs = lr``, so SWA is a running mean of the weights
at the epoch starts, as Lightning's callback samples them),
final ``weights.pt`` = plain state dict with the reference's parameter names (:312). Lightning itself is not used:
the step is ``CryoVITHeadTrainerB200.train_step`` (native forward / backward / all-reduce / AdamW)."""
from __future__ import annotations

import logging
import os
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np
import torch

from ..train import CryoVITHeadTrainerB200
from .datasets import ResidentTomoCache, TomoDataset
from .shard import rank_world, require_process_group


def _cache_budget_bytes(cache_gb: float | None) -> int:
    """HBM the resident training set may take: ``cache_gb`` (``CRYOVIT_B200_FEATURE_CACHE_GB`` when None; 0 disables),
    by default 60 % of what is free on the device right now (the trainer's own buffers for a full-size crop are ~6 GB)."""
    if cache_gb is None:
        env = os.environ.get("CRYOVIT_B200_FEATURE_CACHE_GB", "").strip()
        cache_gb = float(env) if env else None
    if cache_gb is not None:
        return int(cache_gb * 1e9)
    free, _total = torch.cuda.mem_get_info()
    return int(0.6 * free)


def _append_row(path: Path, row: dict, first: bool) -> None:
    """One csv row (a header first), flushed to the file before the next epoch starts."""
    path.parent.mkdir(parents=True, exist_ok=True)
    with open(path, "w" if first else "a") as f:
        if first:
            f.write(",".join(row) + "\n")
        f.write(",".join(str(v) for v in row.values()) + "\n")
        f.flush()


def fit_head(dataset: TomoDataset, in_channels: int = 1536, max_epochs: int = 50, lr: float = 1e-4, weight_decay: float = 1e-3,
             swa_epoch_start: int | None = 40, seed: int = 42, exp_dir: Path | str | None = None, state_dict: dict | None = None,
             log_every: int = 10, cache_gb: float | None = None, epoch_seconds: list | None = None, validator=None,
             val_history: list | None = None) -> dict[str, torch.Tensor]:
    """Trains on the items of ``dataset`` (``train=True`` gives the reference's random 128 x 32 x 32 feature crops);
    with several ranks (torchrun) every rank walks its own round-robin share of a common shuffled order and the
    gradients are averaged over the ranks each step. Returns the final (SWA-averaged if enabled) state dict.

    The tomograms this rank trains on stay resident in HBM after their first read (:class:`ResidentTomoCache`, up to
    ``cache_gb``), and the next item's file read (first epoch) and crop draw happen on a helper thread under the current
    step; crops and order are those of the plain ``dataset[i]`` loop. ``epoch_seconds`` (a list) receives the wall clock of
    every epoch's training, device work included.

    ``validator`` (a :class:`~cryovit_b200.host.validate.Validator`): after the training steps of every epoch it schedules,
    the validation tomograms are scored with the current (not SWA-averaged) weights, as Lightning's ``fit`` does. Its
    resident tomograms share the HBM budget, after the training set's. Rank 0 appends a row per validated epoch to
    ``<exp_dir>/validation.csv``; ``val_history`` (a list) receives the same rows as dicts."""
    rank, world = rank_world()
    require_process_group("fit_head")  # the data is sharded by rank below: the gradients must really be exchanged
    torch.manual_seed(seed)
    np.random.seed(seed + rank)  # crops differ per rank, the shuffled ORDER (below) does not
    # the initial weights follow the seed (the reference's seed_everything(cfg.random_seed)) and are identical on
    # every rank
    trainer = CryoVITHeadTrainerB200(in_channels, lr=lr, weight_decay=weight_decay, state_dict=state_dict, seed=seed)
    order_rng = np.random.default_rng(seed)
    swa_avg, swa_n = None, 0
    step = 0
    cache = None
    cacheable = hasattr(dataset, "_crop_slices") and hasattr(dataset, "_load_tomogram")
    budget = _cache_budget_bytes(cache_gb) if cacheable or validator is not None else 0
    if cacheable:
        if budget > 0:
            cache = ResidentTomoCache(dataset, trainer.device, budget)  # where the trainer lives
    # the helper thread does host work only (file read, crop draw): the trainer captures CUDA graphs on this thread, and a
    # CUDA call from another thread during a capture is an error. ONE helper thread: the crop draws stay in order.
    fetch = (lambda i: cache.prepare(int(i))) if cache is not None else (lambda i: dataset[int(i)])
    pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix="cryovit-fit-fetch")
    val_rows = 0
    try:
        for epoch in range(max_epochs):
            # Lightning's StochasticWeightAveraging.on_train_epoch_START: epochs swa_start .. max_epochs - 1 each add the
            # weights they START from to the running mean (so the last epoch's own updates are not in it), and the mean
            # replaces the weights when training ends.
            if swa_epoch_start is not None and epoch >= swa_epoch_start:
                swa_n += 1
                swa_avg = trainer.flat_p.clone() if swa_avg is None else swa_avg + (trainer.flat_p - swa_avg) / swa_n
            t_epoch = time.perf_counter()
            order = order_rng.permutation(len(dataset))
            usable = len(order) // world * world  # every rank takes the same number of steps (the all-reduce is collective)
            losses = []
            mine = [int(i) for i in order[:usable][rank::world]]
            nxt = pool.submit(fetch, mine[0]) if mine else None
            for k in range(len(mine)):
                item = cache.finish(nxt.result()) if cache is not None else nxt.result()
                nxt = pool.submit(fetch, mine[k + 1]) if k + 1 < len(mine) else None
                dev = trainer.device
                loss = trainer.train_step(item.data.to(dev, non_blocking=True), item.label.to(dev, non_blocking=True))
                step += 1
                if step % log_every == 0 or len(losses) == 0:
                    losses.append(float(loss))
            if rank == 0 or epoch_seconds is not None:
                if torch.device(trainer.device).type == "cuda":
                    torch.cuda.synchronize()
                if epoch_seconds is not None:
                    epoch_seconds.append(time.perf_counter() - t_epoch)
            if rank == 0:
                logging.info("epoch %d: %d steps/rank, DiceLoss %.4f, %.2f s", epoch, usable // world,
                             float(np.mean(losses)) if losses else float("nan"), time.perf_counter() - t_epoch)
            if validator is not None and validator.scheduled(epoch):
                row = validator.run(trainer, epoch, cache_budget=budget - (cache.used if cache is not None else 0))
                if val_history is not None:
                    val_history.append(row)
                if exp_dir is not None and rank == 0:
                    _append_row(Path(exp_dir) / "validation.csv", row, first=val_rows == 0)
                val_rows += 1
    finally:
        pool.shutdown(wait=True)
    if cache is not None and rank == 0:
        logging.info("resident training set: %d tomograms, %.2f GB in HBM, %d file reads for %d steps", len(cache._items),
                     cache.used / 1e9, cache.file_reads, step)
    if swa_avg is not None:
        trainer.flat_p.copy_(swa_avg)
    sd = trainer.state_dict()
    if exp_dir is not None and rank == 0:
        Path(exp_dir).mkdir(parents=True, exist_ok=True)
        torch.save(sd, Path(exp_dir) / "weights.pt")
    return sd
