"""Kernel operands rebuilt from a flat fp32 parameter bucket by ONE gather per output dtype.

Every operand the head's kernels read (tap-major weights, shared-memory images, flipped / transposed copies, repeated
bias tables) is a pure re-arrangement of parameters with zero padding. Running the re-arrangement once on the
parameters' GLOBAL INDICES (index + 1 in fp32, exact up to 2^24) instead of their values turns it into a gather table;
from then on ``index_select`` over the bucket plus one cast rebuild every operand, whatever the number of small torch
kernels the re-arrangement took. The trainer refreshes its bf16 operands this way every step
(``CryoVITHeadTrainerB200._pk``), the inference head all of its operands from the trainer's bucket
(``CryoVITHeadB200.attach_bucket``)."""
from __future__ import annotations

import torch

_ALIGN = 64  # every operand starts 64 elements into its dtype's gathered buffer: >= 128 bytes, what TMA needs and more


class OperandGather:
    def __init__(self, store: torch.Tensor, retired: list | None = None):
        """``store``: fp32 [n + 1], the n parameters and a zero every padding entry reads. ``retired`` (optional) keeps
        superseded concatenated tables alive (a captured CUDA graph gathers through the table it was captured with)."""
        self.store = store
        self.n = store.numel() - 1
        self.tables: dict = {}  # operand name -> (gather table into store, shape, dtype)
        self.views: dict = {}   # operand name -> the operand of the last refresh()
        self._cat = None        # dtype -> (names, concatenated table)
        self._retired = retired

    def indices(self, offset: int, shape, device=None) -> torch.Tensor:
        """The index-valued stand-in of the parameter that starts at ``offset`` in the bucket: fp32, global index + 1
        (0 is what zero padding of the re-arrangement produces)."""
        numel = 1
        for s in shape:
            numel *= s
        dev = self.store.device if device is None else device
        return (torch.arange(numel, device=dev, dtype=torch.float32) + float(offset + 1)).view(tuple(shape))

    def add(self, name: str, t: torch.Tensor, dtype: torch.dtype) -> None:
        """Registers operand ``name`` = the re-arrangement ``t`` of index-valued stand-ins, gathered as ``dtype``."""
        table = t.round().long().flatten().to(self.store.device) - 1
        table[table < 0] = self.n  # padding -> the zero slot
        pad = -table.numel() % _ALIGN
        if pad:
            table = torch.cat([table, torch.full((pad,), self.n, device=table.device, dtype=table.dtype)])
        self.tables[name] = (table, tuple(t.shape), dtype)
        if self._cat is not None and self._retired is not None:
            self._retired.append(self._cat)
        self._cat = None

    def refresh(self) -> dict:
        """One ``index_select`` and one cast per dtype for every registered operand; returns ``name -> operand``."""
        self.views = {}
        if not self.tables:
            return self.views
        if self._cat is None:
            groups: dict = {}
            for name, (_, _, dtype) in self.tables.items():
                groups.setdefault(dtype, []).append(name)
            self._cat = {dt: (names, torch.cat([self.tables[k][0] for k in names])) for dt, names in groups.items()}
        for dt, (names, cat) in self._cat.items():
            packed = self.store.index_select(0, cat).to(dt)
            off = 0
            for k in names:
                table, shape, _ = self.tables[k]
                numel = 1
                for s in shape:
                    numel *= s
                self.views[k] = packed[off:off + numel].view(shape)
                off += table.numel()
        return self.views
