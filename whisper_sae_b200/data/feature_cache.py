"""On-disk activation cache with the reference's interface and file formats
(``whisper_sae.data.feature_cache``, /root/reference/src/whisper_sae/data/feature_cache.py:23-197).

Files (byte-compatible with the reference, so caches are interchangeable):
  ``{model_short}_{component}_layer{N}.pt``        one float32 tensor [num_tokens, d_model]
                                                   (bfloat16 / float16 when extracted with ``dtype=``)
  ``{model_short}_{component}_layer{N}_meta.json`` the 8 ``CacheMetadata`` fields

``get_dataloader`` keeps the reference signature and default behaviour (a ``DataLoader`` over a
``TensorDataset``).  Passing ``device=`` (extension, default off) returns a ``ResidentBatches``
iterable instead: the whole activation matrix lives in pinned host memory or HBM and batches are
cut by a device-side permutation — the per-row Python collate of the stock loader caps out near
1e5-1e6 rows/s, far below what the fused train step consumes.
"""

from __future__ import annotations

import json
from dataclasses import dataclass, fields
from datetime import datetime
from pathlib import Path
from typing import Iterator, Literal

import torch
from torch import Tensor
from torch.utils.data import DataLoader, TensorDataset

from ..config import DataConfig, WhisperConfig

Component = Literal["encoder", "decoder"]


def _jsonable(value):
    if isinstance(value, Path):
        return str(value)
    if isinstance(value, dict):
        return {k: _jsonable(v) for k, v in value.items()}
    return value


@dataclass
class CacheMetadata:
    """Sidecar description of one cached layer (feature_cache.py:23-57)."""

    model_name: str
    component: Component
    layer_idx: int
    hidden_dim: int
    num_samples: int
    num_tokens: int
    created_at: str
    data_config: dict

    def to_json(self) -> str:
        return json.dumps({f.name: _jsonable(getattr(self, f.name)) for f in fields(self)}, indent=2)

    @classmethod
    def from_json(cls, json_str: str) -> "CacheMetadata":
        return cls(**json.loads(json_str))


class IndexedBatch:
    """A batch named by reference: rows ``rows`` (int64, device) of the resident ``features`` matrix.

    What the reference's ``DataLoader(TensorDataset(features), shuffle=True)`` materialises per step
    (feature_cache.py:169-197) - here the graphed train step reads the rows where they lie (K0 and
    K23 take the matrix address and the index array from device slots: ``wsae_pack_activations_rows_at``,
    ``wsae_decode_backward_rows_at``), so a shuffled epoch costs no gather pass (233 MB of HBM traffic
    per 75 776-row batch at d = 384).  ``materialize()`` gives the plain tensor for every other consumer.
    """

    __slots__ = ("features", "rows")

    def __init__(self, features: Tensor, rows: Tensor):
        if features.dim() != 2 or rows.dim() != 1 or rows.dtype != torch.int64:
            raise ValueError("IndexedBatch needs a [N, d] matrix and a 1-d int64 row-index tensor")
        self.features = features
        self.rows = rows

    @property
    def shape(self) -> torch.Size:
        return torch.Size((self.rows.shape[0], self.features.shape[1]))

    @property
    def dtype(self) -> torch.dtype:
        return self.features.dtype

    @property
    def device(self) -> torch.device:
        return self.features.device

    @property
    def is_cuda(self) -> bool:
        return self.features.is_cuda

    def dim(self) -> int:
        return 2

    def __len__(self) -> int:
        return self.rows.shape[0]

    def materialize(self) -> Tensor:
        return self.features.index_select(0, self.rows)

    def to(self, *args, **kwargs) -> Tensor:
        return self.materialize().to(*args, **kwargs)


class ResidentBatches:
    """Batches cut from a resident [N, d] matrix by a device-side permutation each epoch.  On a CUDA
    device a shuffled batch is an :class:`IndexedBatch` (matrix + slice of the permutation): the train
    step gathers the rows inside its own kernels instead of an ``index_select`` pass per batch."""

    def __init__(self, features: Tensor, batch_size: int, shuffle: bool, device: torch.device | str,
                 drop_last: bool = False, seed: int | None = None, indexed: bool | None = None):
        self.features = features.to(device)
        self.batch_size = batch_size
        self.shuffle = shuffle
        self.drop_last = drop_last
        self.indexed = self.features.is_cuda if indexed is None else bool(indexed)
        self._gen = torch.Generator(device=self.features.device)
        if seed is not None:
            self._gen.manual_seed(seed)

    def __len__(self) -> int:
        n = self.features.shape[0]
        return n // self.batch_size if self.drop_last else (n + self.batch_size - 1) // self.batch_size

    def __iter__(self) -> Iterator[list]:
        n = self.features.shape[0]
        order = (torch.randperm(n, device=self.features.device, generator=self._gen)
                 if self.shuffle else None)
        for i in range(len(self)):
            lo, hi = i * self.batch_size, min(n, (i + 1) * self.batch_size)
            if order is None:
                rows = self.features[lo:hi]
            elif self.indexed:
                rows = IndexedBatch(self.features, order[lo:hi])
            else:
                rows = self.features.index_select(0, order[lo:hi])
            yield [rows]  # same 1-element list a TensorDataset loader yields


class FeatureCache:
    """Per-layer activation cache (feature_cache.py:60-197)."""

    def __init__(self, cache_dir: Path, whisper_config: WhisperConfig, data_config: DataConfig):
        self.cache_dir = Path(cache_dir)
        self.cache_dir.mkdir(parents=True, exist_ok=True)
        self.whisper_config = whisper_config
        self.data_config = data_config
        self.model_short = whisper_config.model_name.split("/")[-1]

    def _stem(self, component: Component, layer_idx: int) -> str:
        return f"{self.model_short}_{component}_layer{layer_idx}"

    def _get_cache_path(self, component: Component, layer_idx: int) -> Path:
        return self.cache_dir / f"{self._stem(component, layer_idx)}.pt"

    def _get_metadata_path(self, component: Component, layer_idx: int) -> Path:
        return self.cache_dir / f"{self._stem(component, layer_idx)}_meta.json"

    def has_cache(self, component: Component, layer_idx: int) -> bool:
        return (self._get_cache_path(component, layer_idx).exists()
                and self._get_metadata_path(component, layer_idx).exists())

    def load(self, component: Component, layer_idx: int) -> tuple[Tensor, CacheMetadata]:
        """The cached matrix in its stored dtype (a bf16 / fp16 cache stays half precision: the graphed
        train step reads it in place) and its metadata."""
        features = torch.load(self._get_cache_path(component, layer_idx), weights_only=True)
        meta = CacheMetadata.from_json(self._get_metadata_path(component, layer_idx).read_text())
        return features, meta

    def save(self, features: Tensor, component: Component, layer_idx: int, num_samples: int) -> None:
        torch.save(features, self._get_cache_path(component, layer_idx))
        meta = CacheMetadata(
            model_name=self.whisper_config.model_name,
            component=component,
            layer_idx=layer_idx,
            hidden_dim=features.shape[-1],
            num_samples=num_samples,
            num_tokens=features.shape[0],
            created_at=datetime.now().isoformat(),
            data_config=self.data_config.model_dump(),
        )
        self._get_metadata_path(component, layer_idx).write_text(meta.to_json())

    def get_dataloader(self, component: Component, layer_idx: int, batch_size: int,
                       shuffle: bool = True, num_workers: int = 0, *,
                       device: torch.device | str | None = None):
        """Batches of the cached matrix in its stored dtype; a bf16 / fp16 cache trains in place."""
        features, _ = self.load(component, layer_idx)
        if device is not None:
            return ResidentBatches(features, batch_size, shuffle, device)
        return DataLoader(TensorDataset(features), batch_size=batch_size, shuffle=shuffle,
                          num_workers=num_workers, pin_memory=True)


def extract_and_cache_features(whisper_model, processor, audio_dataloader, cache: FeatureCache,
                               encoder_layers: list[int], decoder_layers: list[int],
                               device: torch.device | str = "cuda",
                               max_samples: int | None = None, *,
                               device_budget_bytes: int = 8 << 30,
                               dtype: torch.dtype = torch.float32) -> None:
    """Run Whisper over ``audio_dataloader`` and write one cache file per hooked layer
    (feature_cache.py:200-306; same signature, ``processor`` is unused there too).

    Hooked hidden states are normalised (the model's final LayerNorm) and flattened straight into a
    growable device matrix per layer (``sae.hooks.ActivationMatrix``); nothing visits the host until
    ``cache.save`` writes the ``[N, d]`` fp32 tensor in the reference's file format - unless the
    hooked layers together would hold more than ``device_budget_bytes`` on the GPU, in which case full
    chunks are spilled to pinned host memory as they fill (the reference accumulates on the host).

    ``dtype`` (extension): ``torch.bfloat16`` or ``torch.float16`` writes half-precision cache files,
    the fp32 LayerNorm result rounded to nearest - half the bytes on disk, in host memory, on PCIe and
    in HBM.  The file format and the metadata are otherwise unchanged; ``SAETrainer`` trains on such a
    matrix in place, while the reference's trainer needs ``.float()`` to read it.
    """
    if dtype not in (torch.float32, torch.bfloat16, torch.float16):
        raise ValueError(f"cache dtype must be float32, bfloat16 or float16, not {dtype}")
    from ..sae.hooks import ActivationMatrix, _hidden_of, run_whisper

    whisper_model = whisper_model.to(device)
    whisper_model.eval()
    d = whisper_model.config.d_model
    n_sinks = max(1, len(encoder_layers) + len(decoder_layers))
    elem = torch.empty((), dtype=dtype).element_size()
    cap_rows = max(4096, device_budget_bytes // (n_sinks * d * elem))
    enc = {layer: ActivationMatrix(d, device, max_device_rows=cap_rows, dtype=dtype) for layer in encoder_layers}
    dec = {layer: ActivationMatrix(d, device, max_device_rows=cap_rows, dtype=dtype) for layer in decoder_layers}
    enc_ln, dec_ln = whisper_model.model.encoder.layer_norm, whisper_model.model.decoder.layer_norm
    handles = []
    for layer, sink in enc.items():
        handles.append(whisper_model.model.encoder.layers[layer].register_forward_hook(
            lambda m, i, o, sink=sink: sink.append(_hidden_of(o).detach(), enc_ln)))
    for layer, sink in dec.items():
        handles.append(whisper_model.model.decoder.layers[layer].register_forward_hook(
            lambda m, i, o, sink=sink: sink.append(_hidden_of(o).detach(), dec_ln)))
    num_samples = 0
    target = max_samples if max_samples is not None else float("inf")
    try:
        with torch.no_grad():
            for batch in audio_dataloader:
                if num_samples >= target:
                    break
                if isinstance(batch, (list, tuple)):
                    batch = batch[0]
                batch = batch.to(device)
                run_whisper(whisper_model, batch, bool(decoder_layers))
                num_samples += batch.shape[0]
    finally:
        for h in handles:
            h.remove()
    for component, sinks in (("encoder", enc), ("decoder", dec)):
        for layer, sink in sinks.items():
            if sink.rows:
                cache.save(sink.tensor().cpu(), component, layer, num_samples)
