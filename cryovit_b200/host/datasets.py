"""Datasets and batch assembly on either side of the hot path, with the reference's semantics.

``VITDataset``  (datasets/vit_dataset.py:23-123): one tomogram per item for feature extraction.
``TomoDataset`` (datasets/tomo_dataset.py:20-178) + ``collate_fn`` (datamodules/utils.py:13-121): feature volume +
labels for the head, with the training crop.
"""
from __future__ import annotations

import logging
from dataclasses import dataclass, field
from pathlib import Path
from typing import Any

import numpy as np
import torch

from .. import ops
from .._lib import CryovitB200Error
from . import hdf


class VITDataset:
    """``VITDataset(data_root, use_sam, records)``; item i is tomogram ``records[i]``.

    ``fused=True`` (default) returns the RAW tomogram ``[D, H, W]`` (uint8, or float32 in [0,1]) so that the
    pre-processing of ``_dino_transform`` runs inside the GPU extractor and 1 byte per voxel crosses PCIe.
    ``fused=False`` keeps the reference's item exactly: float32 ``[D, 3, H', W']`` (pad-to-16 edge, three identical
    channels, bicubic x14/16), computed by the sm_100a resize kernel on the current CUDA device and returned on the
    host, as the reference's dataset does. The ImageNet ``Normalize`` the reference constructs is never applied
    there (vit_dataset.py:39 vs :90-123), so it does not exist here.
    """

    def __init__(self, data_root: Path | str, use_sam: bool = False, records: list[str] | None = None, fused: bool = True):
        if use_sam:
            raise CryovitB200Error("use_sam=True (SAM2 image encodings) is outside the B200 hot path")
        self.root = Path(data_root)
        self.use_sam = use_sam
        self.records = list(records or [])
        self.fused = fused
        self._warned = False

    def __len__(self) -> int:
        return len(self.records)

    def _load_tomogram(self, record: str) -> np.ndarray:
        """vit_dataset.py:71-88 reads ``data``; the uint8 -> /255 conversion happens in the GPU kernel."""
        data = hdf.read_tomogram(self.root / record, keys=["data"])["data"]
        if data.dtype not in (np.uint8, np.float32):
            data = data.astype(np.float32)
        return data

    def __getitem__(self, idx: int) -> torch.Tensor:
        if idx >= len(self):
            raise IndexError
        return self.item_from_array(self._load_tomogram(self.records[idx]))

    def item_from_array(self, data: np.ndarray) -> torch.Tensor:
        """The item for a ``data`` array that is already in memory (the feature runner reads each source file once
        and passes its ``data`` both here and through to the result file)."""
        if data.dtype not in (np.uint8, np.float32):
            data = data.astype(np.float32)
        _, h, w = data.shape
        if (h % 16 or w % 16) and not self._warned:
            logging.warning("Resizing tomogram from %s to %s", (h, w), ((h + 15) // 16 * 16, (w + 15) // 16 * 16))
            self._warned = True
        t = torch.from_numpy(np.ascontiguousarray(data))
        if self.fused:
            return t
        dev = t.cuda(non_blocking=True)
        OH, OW, _, _ = ops.patch_grid(h, w)
        out = torch.empty(t.shape[0], 3, OH, OW, device=dev.device, dtype=torch.float32)
        ops.preproc_resize_3ch(dev, out)
        return out.cpu()


@dataclass
class TomogramData:
    """types.py TomogramData: one tomogram for the head (data ``[C, D, h, w]``, label ``[D, H, W]``)."""

    sample: str
    tomo_name: str
    split_id: int | None
    data: torch.Tensor
    label: torch.Tensor
    aux_data: dict[str, Any] = field(default_factory=dict)


@dataclass
class BatchedTomogramMetadata:
    samples: list[str]
    tomo_names: list[str]
    unique_id: torch.Tensor
    split_id: torch.Tensor | None

    def identifiers(self) -> tuple[list[str], list[str]]:
        return ([self.samples[int(i[0])] for i in self.unique_id], [self.tomo_names[int(i[1])] for i in self.unique_id])


@dataclass
class BatchedTomogramData:
    """types.py BatchedTomogramData as a plain dataclass (tensordict is not a dependency here)."""

    tomo_batch: torch.Tensor   # [B, D, C, h, w]
    tomo_sizes: torch.Tensor   # [B]
    labels: torch.Tensor       # [B, D, H, W], -1 = ignore
    metadata: BatchedTomogramMetadata
    min_slices: int
    aux_data: dict[str, list[Any]] | None = None

    @property
    def num_tomos(self) -> int:
        return self.tomo_batch.shape[0]

    @property
    def num_slices(self) -> int:
        return self.tomo_batch.shape[1]

    def pin_memory(self, device=None):
        self.tomo_batch = self.tomo_batch.pin_memory()
        self.tomo_sizes = self.tomo_sizes.pin_memory()
        self.labels = self.labels.pin_memory()
        return self


class TomoDataset:
    """Feature volume + label of one tomogram per item (datasets/tomo_dataset.py). ``records`` is anything with
    ``.iloc[i]`` rows holding ``sample`` and ``tomo_name`` (a pandas DataFrame), or a list of dicts."""

    def __init__(self, records, input_key: str, label_key: str, split_key: str, data_root: Path | str,
                 aux_keys: list[str] | None = None, train: bool = False, rng: np.random.Generator | None = None):
        self.records = records
        self.input_key, self.label_key, self.split_key = input_key, label_key, split_key
        self.aux_keys = list(aux_keys or [])
        self.data_root = Path(data_root)
        self.train = train
        self.rng = rng  # None: numpy's global generator, as the reference (np.random.choice)

    def __len__(self) -> int:
        return len(self.records)

    def _row(self, idx: int) -> dict:
        r = self.records.iloc[idx] if hasattr(self.records, "iloc") else self.records[idx]
        return dict(r)

    def _load_tomogram(self, record: dict) -> dict[str, Any]:
        path = self.data_root / record["sample"] / record["tomo_name"]
        keys = hdf.list_keys(path)
        if self.input_key not in keys:
            raise CryovitB200Error(f"Input key '{self.input_key}' not found in {path}.")
        if f"labels/{self.label_key}" not in keys:
            raise CryovitB200Error(f"Label key '{self.label_key}' not found in {path}/labels.")
        want = [self.input_key, f"labels/{self.label_key}"] + [k for k in self.aux_keys if k in keys]
        got = hdf.read_tomogram(path, keys=want)
        data = got[self.input_key]
        if data.dtype == np.uint8:
            data = data.astype(np.float32) / 255.0
        if data.ndim == 3:
            data = data[np.newaxis]
        out = {"sample": record["sample"], "tomo_name": record["tomo_name"], "input": data,
               "label": got[f"labels/{self.label_key}"]}
        if self.split_key in record:
            out["split_id"] = record[self.split_key]
        for k in self.aux_keys:
            if k in got:
                out[k] = got[k]
        return out

    def max_crop_shape(self) -> tuple[int, int, int]:
        """(depth, rows, cols) of the largest input crop ``_crop_slices`` cuts: at most 128 slices, 32x32 feature patches
        (512x512 voxels for raw input)."""
        side = 32 if self.input_key == "dino_features" else 512
        return 128, side, side

    def _crop_slices(self, shape) -> tuple[tuple[slice, ...], tuple[slice, ...]] | None:
        """tomo_dataset.py:148-178: at most 128 slices, 32x32 feature patches (512x512 voxels for raw input); the
        label crop is the x16 image of the feature crop. Draw order (depth, rows, cols) follows the reference. Only
        the SHAPE is needed, so the same draw serves a numpy array from a file and a volume resident in HBM.
        Returns (input slices over the last three axes, label slices) or None when nothing is cropped."""
        max_depth, side, _ = self.max_crop_shape()
        d, h, w = shape[-3:]
        x, y, z = min(d, max_depth), side, side
        if (d, h, w) == (x, y, z):
            return None
        choice = self.rng.choice if self.rng is not None else np.random.choice
        dd, dh, dw = d - x + 1, h - y + 1, w - z + 1
        di = int(choice(dd)) if dd > 0 else 0
        hi = int(choice(dh)) if dh > 0 else 0
        wi = int(choice(dw)) if dw > 0 else 0
        inp = (slice(di, di + x), slice(hi, hi + y), slice(wi, wi + z))
        if self.input_key == "dino_features":
            hi, wi, y, z = 16 * hi, 16 * wi, 16 * y, 16 * z
        return inp, (slice(di, di + x), slice(hi, hi + y), slice(wi, wi + z))

    def _random_crop(self, data: dict[str, Any]) -> None:
        crop = self._crop_slices(data["input"].shape)
        if crop is not None:
            data["input"] = data["input"][(..., *crop[0])]
            data["label"] = data["label"][crop[1]]

    def __getitem__(self, idx: int) -> TomogramData:
        if idx >= len(self):
            raise IndexError
        rec = self._row(idx)
        data = self._load_tomogram(rec)
        if self.train:
            self._random_crop(data)
        return TomogramData(sample=rec["sample"], tomo_name=rec["tomo_name"], split_id=data.get("split_id"),
                            data=torch.as_tensor(np.ascontiguousarray(data["input"])),
                            label=torch.as_tensor(np.ascontiguousarray(data["label"])),
                            aux_data={k: data[k] for k in self.aux_keys if k in data})


class ResidentTomoCache:
    """The training set kept where the head trains: whole (uncropped) feature volumes and labels of a ``TomoDataset``
    on ``device``, loaded from their files once. The reference re-reads every tomogram file in every epoch
    (tomo_dataset.py:89-146 under a 50-epoch fit, configs/trainer/fit.yaml): 403 MB of features per step against a
    19 ms step. A B200 holds 180 GB: ~400 tomograms of BASELINE's size fit next to the trainer. ``get(i)`` is
    ``dataset[i]`` with the tensors already on the device: same record order, same crop draws (the crop is drawn from
    the shape and applied as a view of the resident volume). Items past ``budget_bytes`` are not kept and come from
    their file every time, as before.

    ``int8_labels`` (validation): a label volume whose values are all in {-1, 0, 1} is kept as int8, the operand of
    ``CryoVITHeadB200.score_volume``'s fused path (a quarter of fp32's HBM); the values are checked once per file read,
    and other labels stay as they are."""

    def __init__(self, dataset: "TomoDataset", device, budget_bytes: int, int8_labels: bool = False):
        self.dataset, self.device, self.budget = dataset, torch.device(device), int(budget_bytes)
        self.int8_labels = int8_labels
        self.used = 0
        self.file_reads = 0
        self._items: dict[int, tuple[torch.Tensor, torch.Tensor, dict]] = {}

    def _load(self, idx: int):
        ds = self.dataset
        rec = ds._row(idx)
        data = ds._load_tomogram(rec)
        self.file_reads += 1
        label = data["label"]
        if self.int8_labels and label.dtype != np.int8 and np.isin(label, (-1, 0, 1)).all():
            label = label.astype(np.int8)
        inp, lab = torch.as_tensor(np.ascontiguousarray(data["input"])), torch.as_tensor(np.ascontiguousarray(label))
        meta = {"sample": rec["sample"], "tomo_name": rec["tomo_name"], "split_id": data.get("split_id"),
                "aux": {k: data[k] for k in ds.aux_keys if k in data}}
        return inp, lab, meta

    def prepare(self, idx: int):
        """Host-only half of :meth:`get` (safe on a helper thread while the main thread captures a CUDA graph: no CUDA
        call here): the file read of a tomogram that is not resident yet, and the crop draw -- from the shape, in call
        order."""
        if idx >= len(self.dataset):
            raise IndexError
        hit = self._items.get(idx)
        loaded = None if hit is not None else self._load(idx)
        shape = (hit or loaded)[0].shape
        crop = self.dataset._crop_slices(shape) if self.dataset.train else None
        return idx, loaded, crop

    def finish(self, prepared) -> TomogramData:
        """Device half (main thread): upload + keep a newly read tomogram if the budget allows, cut the crop as a view."""
        idx, loaded, crop = prepared
        if loaded is not None:
            inp, lab, meta = loaded
            need = inp.numel() * inp.element_size() + lab.numel() * lab.element_size()
            if idx not in self._items and self.used + need <= self.budget:
                inp, lab = inp.to(self.device), lab.to(self.device)
                self._items[idx] = (inp, lab, meta)
                self.used += need
        else:
            inp, lab, meta = self._items[idx]
        if crop is not None:
            inp, lab = inp[(..., *crop[0])], lab[crop[1]]
        return TomogramData(sample=meta["sample"], tomo_name=meta["tomo_name"], split_id=meta["split_id"],
                            data=inp.contiguous(), label=lab.contiguous(), aux_data=meta["aux"])

    def get(self, idx: int) -> TomogramData:
        return self.finish(self.prepare(idx))


def collate_fn(batch: list[TomogramData]) -> BatchedTomogramData:
    """datamodules/utils.py:13-121. Depth is padded to the longest tomogram of the batch: data with 0, labels with
    -1 (ignored by the masked loss). The reference's padding branch pads ``data`` a second time where it means the
    label (:83-85) and would fail on the shape; the intended behaviour is implemented here."""
    sizes = torch.tensor([t.data.shape[-3] for t in batch], dtype=torch.int)
    max_size, min_slices = int(sizes.max()), int(sizes.min())
    C, _, hp, wp = batch[0].data.shape
    H, W = batch[0].label.shape[-2:]
    tomo_batch = torch.zeros(len(batch), C, max_size, hp, wp, dtype=torch.float)
    labels = torch.full((len(batch), max_size, H, W), -1.0, dtype=torch.float)
    aux: dict[str, list] = {k: [] for k in batch[0].aux_data}
    uniq_s: dict[str, None] = {}
    uniq_n: dict[str, None] = {}
    ident = torch.empty(len(batch), 2, dtype=torch.long)
    split = torch.empty(len(batch), dtype=torch.int)
    use_splits = True
    for i, t in enumerate(batch):
        D = t.data.shape[-3]
        tomo_batch[i, :, :D] = t.data.float()
        labels[i, :D] = t.label.float()
        for k, v in t.aux_data.items():
            aux[k].append(v)
        uniq_s[t.sample] = None
        uniq_n[t.tomo_name] = None
        ident[i, 0] = list(uniq_s).index(t.sample)
        ident[i, 1] = list(uniq_n).index(t.tomo_name)
        if t.split_id is not None and use_splits:
            split[i] = int(t.split_id)
        else:
            use_splits = False
    meta = BatchedTomogramMetadata(list(uniq_s), list(uniq_n), ident, split if use_splits else None)
    return BatchedTomogramData(tomo_batch=tomo_batch.permute(0, 2, 1, 3, 4), tomo_sizes=sizes, labels=labels,
                               metadata=meta, min_slices=min_slices, aux_data=aux)
