"""Lightning's validation loop for head training (reference ``trainer.fit(model, datamodule)``, run/train_model.py:
300-310, with models/base_model.py:130-148 ``validation_step`` and configs/model/default.yaml's losses and metrics).

After the training steps of every scheduled epoch, each validation tomogram (the held-out ``split_id``, or the
training set when there is none: ``val_df()``) is scored WHOLE with the current weights, batch size one as in the
reference: every loss and metric is the mean over tomograms of its per-tomogram value. The scoring runs inside the
output convolution (``CryoVITHeadB200.score_volume``), the inference head takes the trainer's weights straight from
its flat parameter bucket (``CryoVITHeadB200.attach_bucket`` / ``refresh``) and the tomograms stay resident in HBM
(``ResidentTomoCache``, labels as int8) next to the training set. Nothing here draws from numpy's or torch's global
random generators, so the trained weights are the same with validation on or off.

Not modelled: Lightning's pre-training sanity check (``num_sanity_val_steps``: it changes no output), the granule
experiments' mito mask, early stopping and best-checkpoint selection (the reference configures neither)."""
from __future__ import annotations

import logging
import time

import torch

from ..head import CryoVITHeadB200
from .datasets import ResidentTomoCache
from .metrics import DiceLoss, DiceMetric, F1Metric, SegStats, _MeanOfBatchesMetric
from .shard import rank_world, shard_round_robin


def val_schedule(check_val_every_n_epoch=1, limit_val_batches=1.0, n_tomograms: int = 0) -> tuple[int, int]:
    """Lightning's rules for the two trainer keys -> (validate every n-th epoch: epoch e when (e + 1) % n == 0, the
    number of validation tomograms). ``limit_val_batches``: an int is a count (capped at the set), a float in [0, 1] a
    fraction of the set (1.0: all), 0 disables validation; a nonzero fraction that leaves no tomogram is an error, as
    in Lightning."""
    n = check_val_every_n_epoch
    if isinstance(n, bool) or not isinstance(n, int) or n < 1:
        raise ValueError(f"trainer.check_val_every_n_epoch must be an int >= 1, got {n!r}")
    lim = limit_val_batches
    if isinstance(lim, bool) or not isinstance(lim, (int, float)):
        raise ValueError(f"trainer.limit_val_batches must be an int or a float, got {lim!r}")
    if isinstance(lim, int):
        if lim < 0:
            raise ValueError(f"trainer.limit_val_batches must be >= 0, got {lim}")
        return n, min(n_tomograms, lim)
    if not 0.0 <= lim <= 1.0:
        raise ValueError(f"trainer.limit_val_batches as a float is a fraction in [0, 1], got {lim}")
    count = int(n_tomograms * lim)
    if count == 0 and lim > 0.0 and n_tomograms > 0:
        raise ValueError(f"trainer.limit_val_batches={lim} of {n_tomograms} validation tomograms is less than one; "
                         f"use at least {1.0 / n_tomograms}")
    return n, count


class Validator:
    """The validation set of a head training run, its resident cache, the inference head that follows the trainer,
    and the losses and metrics of ``cfg.model`` (``DiceLoss``, ``DiceMetric``, ``F1Metric``: the ones the reference's
    configs name; anything else is refused here)."""

    def __init__(self, dataset, in_channels: int, losses: dict, metrics: dict, check_val_every_n_epoch=1,
                 limit_val_batches=1.0):
        for k, fn in losses.items():
            if not isinstance(fn, DiceLoss):
                raise ValueError(f"validation: loss {k!r} ({type(fn).__name__}) is not supported; DiceLoss is")
        for k, m in metrics.items():
            if not isinstance(m, (DiceMetric, F1Metric)):
                raise ValueError(f"validation: metric {k!r} ({type(m).__name__}) is not supported; DiceMetric and F1Metric are")
        self.dataset, self.in_channels = dataset, in_channels
        self.losses, self.metrics = dict(losses), dict(metrics)
        self.every, self.count = val_schedule(check_val_every_n_epoch, limit_val_batches, len(dataset))
        self.head = None
        self.cache = None

    def scheduled(self, epoch: int) -> bool:
        return self.count > 0 and (epoch + 1) % self.every == 0

    def _thresholds(self) -> list[float]:
        """The thresholds the sums must be taken at: 0.5 (DiceLoss and F1Metric read only threshold-free sums and the
        strict p > 0.5 ones) and every DiceMetric's own."""
        out = [0.5]
        for m in self.metrics.values():
            if isinstance(m, DiceMetric) and float(m.threshold) not in out:
                out.append(float(m.threshold))
        return out

    def run(self, trainer, epoch: int, cache_budget: int = 0) -> dict:
        """Scores this rank's share (round robin) of the first ``count`` validation tomograms with the trainer's current
        weights; every rank must call it (the states are summed over the ranks). ``cache_budget``: HBM bytes the
        validation tomograms may keep (taken on the first call). Returns the row
        ``{epoch, <loss keys>, <metric keys>, tomograms, seconds}``."""
        t0 = time.perf_counter()
        dev = trainer.device
        if self.head is None:
            self.head = CryoVITHeadB200(self.in_channels).cuda(dev.index).attach_bucket(*trainer.parameter_bucket())
            if hasattr(self.dataset, "_load_tomogram"):
                self.cache = ResidentTomoCache(self.dataset, dev, max(0, int(cache_budget)), int8_labels=True)
        else:
            self.head.refresh()
        loss_means = {k: _MeanOfBatchesMetric() for k in self.losses}
        for m in self.metrics.values():
            m.reset()
        thresholds = self._thresholds()
        for i in shard_round_robin(list(range(self.count))):
            item = self.cache.get(i) if self.cache is not None else self.dataset[i]
            feats, labels = item.data.to(dev, non_blocking=True), item.label.to(dev, non_blocking=True)
            stats = {t: SegStats.from_sums(self.head.score_volume(feats, labels, t)) for t in thresholds}
            for k, fn in self.losses.items():
                loss_means[k]._add(fn.from_stats(stats[0.5]))
            for m in self.metrics.values():
                m.update_stats(stats[float(m.threshold)] if isinstance(m, DiceMetric) else stats[0.5])
        for m in list(loss_means.values()) + list(self.metrics.values()):
            m.all_reduce(device=dev)
        row = {"epoch": epoch}
        row.update({k: float(m.compute()) for k, m in loss_means.items()})
        row.update({k: float(m.compute()) for k, m in self.metrics.items()})
        row["tomograms"] = int(next(iter(loss_means.values())).total) if loss_means else self.count
        torch.cuda.synchronize(dev)
        row["seconds"] = time.perf_counter() - t0
        if rank_world()[0] == 0:
            logging.info("validation epoch %d: %d tomograms, %s, %.2f s", epoch, row["tomograms"],
                         ", ".join(f"{k} {row[k]:.4f}" for k in list(self.losses) + list(self.metrics)), row["seconds"])
        return row
