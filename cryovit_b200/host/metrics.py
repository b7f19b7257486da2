"""Masked loss and metrics of the head (models/base_model.py:91-112, losses.py:17-32, metrics.py:30-93) on top of
ONE fused reduction pass over the volume (``cvit_seg_stats``). Metric objects keep the reference's update /
compute / reset life cycle and its sum-reducible states (``dist_reduce_fx="sum"``, metrics.py:24-27,64-67): a
data-parallel evaluation all-reduces two numbers per metric."""
from __future__ import annotations

import torch

from .. import ops


class SegStats:
    """The eight masked sums of a (probabilities, labels) pair; labels == -1 are ignored."""

    def __init__(self, probs: torch.Tensor, labels: torch.Tensor, threshold: float = 0.5):
        p = probs.reshape(-1).float().contiguous()
        y = labels.reshape(-1).float().contiguous()
        self.v = ops.seg_stats(p, y, threshold)  # fp64 [8] on the device

    @classmethod
    def from_sums(cls, v: torch.Tensor) -> "SegStats":
        """The same object over sums computed elsewhere (``CryoVITHeadB200.score_volume``): fp64 [8] in the order above."""
        st = cls.__new__(cls)
        st.v = v
        return st

    def dice_loss(self) -> torch.Tensor:
        """losses.py:17-32: 1 - 2*sum(y*p) / (sum(y) + sum(p) + 1e-3)."""
        v = self.v
        return 1.0 - 2.0 * v[2] / (v[1] + v[0] + 1e-3)


class DiceLoss:
    def __call__(self, probs: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        return self.from_stats(SegStats(probs, labels))

    def from_stats(self, stats: SegStats) -> torch.Tensor:
        return stats.dice_loss()


class _MeanOfBatchesMetric:
    """The reference's metrics average the per-batch score: states ``score`` and ``total``, both reduced with "sum"."""

    def __init__(self):
        self.score = None
        self.total = 0.0

    def reset(self) -> None:
        self.score, self.total = None, 0.0

    def _add(self, s: torch.Tensor) -> None:
        self.score = s.clone() if self.score is None else self.score + s
        self.total += 1.0

    def compute(self) -> torch.Tensor:
        if self.total <= 0 or self.score is None:
            return torch.tensor(0.0)
        return self.score / self.total

    def all_reduce(self, device=None) -> None:
        """Data-parallel evaluation: sum both states over ranks (torchmetrics' dist_reduce_fx="sum"). ``device``: where a
        rank that saw no batch puts its zeros (NCCL needs the GPU; default CPU)."""
        import torch.distributed as dist

        if dist.is_available() and dist.is_initialized():
            dev = self.score.device if self.score is not None else (device or "cpu")
            st = torch.stack([(self.score if self.score is not None else torch.zeros((), dtype=torch.float64, device=dev)),
                              torch.tensor(self.total, dtype=torch.float64, device=dev)])
            dist.all_reduce(st, op=dist.ReduceOp.SUM)
            self.score, self.total = st[0], float(st[1])


class DiceMetric(_MeanOfBatchesMetric):
    """metrics.py:8-53: hard prediction (p < thr -> 0 else 1); per batch 2*I / (sum y + sum hard + 1e-3)."""

    def __init__(self, threshold: float = 0.5):
        super().__init__()
        self.threshold = threshold

    def update(self, probs, labels) -> None:
        self.update_stats(SegStats(probs, labels, self.threshold))

    def update_stats(self, stats: SegStats) -> None:
        """``stats``: sums taken with this metric's threshold."""
        v = stats.v
        self._add(2.0 * v[3] / (v[1] + v[4] + 1e-3))


class F1Metric(_MeanOfBatchesMetric):
    """metrics.py:56-93: tp / fp / fn with the strict decision p > 0.5; eps 1e-6 in precision, recall and F1."""

    def update(self, probs, labels) -> None:
        self.update_stats(SegStats(probs, labels))

    def update_stats(self, stats: SegStats) -> None:
        v = stats.v
        tp, fp, fn = v[5], v[6], v[7]
        precision = tp / (tp + fp + 1e-6)
        recall = tp / (tp + fn + 1e-6)
        self._add(2.0 * precision * recall / (precision + recall + 1e-6))
