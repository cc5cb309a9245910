"""Whisper activation extraction (reference: sae/hooks.py) — the producer of the activation cache.

Same names and call shapes as the reference's ``ActivationCache`` / ``WhisperActivationExtractor`` /
``extract_features_batch`` / ``flatten_activations``.  Differences, all on the device side:

* hooked hidden states never leave the GPU (the reference copies every one to the host,
  hooks.py:90,107); the model's final LayerNorm (hooks.py:85-86,103-104) is applied by
  ``wsae_layernorm_rows``, which writes fp32 rows and can append them straight into a caller-owned
  ``[N, d]`` activation matrix (:class:`ActivationMatrix`) — flatten + concatenate
  (hooks.py:213-230, feature_cache.py:283-300) are just the destination offset;
* layer outputs are accepted as a tensor or as a tuple: the reference's decoder hook indexes
  ``output[0]`` (hooks.py:101), which under transformers >= 5 (layers return a bare tensor) picks the
  first *sample* instead of the hidden states.

The Whisper forward itself is the library's (transformers + PyTorch): plumbing, not the product.
CUDA only — a model on another device raises.
"""

from __future__ import annotations

from dataclasses import dataclass, field
from typing import Callable, Literal

import torch
from torch import Tensor, nn

from .. import ops


@dataclass
class ActivationCache:
    """Per-layer lists of captured activations (hooks.py:15-37); tensors stay on the device."""

    encoder: dict[int, list[Tensor]] = field(default_factory=dict)
    decoder: dict[int, list[Tensor]] = field(default_factory=dict)

    def clear(self) -> None:
        self.encoder.clear()
        self.decoder.clear()

    @staticmethod
    def _cat(store: dict[int, list[Tensor]], layer: int) -> Tensor | None:
        if not store.get(layer):
            return None
        return torch.cat(store[layer], dim=0)

    def get_encoder_activations(self, layer: int) -> Tensor | None:
        return self._cat(self.encoder, layer)

    def get_decoder_activations(self, layer: int) -> Tensor | None:
        return self._cat(self.decoder, layer)


class ActivationMatrix:
    """Growable ``[N, d]`` matrix (fp32, or bf16 / fp16 with ``dtype=``) that hooked batches are normalised
    INTO, on the device.

    ``max_device_rows`` bounds the device-resident part: when the next batch would not fit, the rows
    gathered so far are spilled to pinned host memory (one D2H copy per spill, the reference copies
    every hooked tensor, hooks.py:90,107) and the device buffer is reused - so a long extraction over
    many layers (1500 encoder tokens per sample) cannot exhaust HBM.  Growth never keeps an old and a
    new buffer alive beyond the copy, and never grows past the bound.
    """

    def __init__(self, d: int, device: torch.device | str, capacity: int = 1 << 16,
                 max_device_rows: int | None = None, dtype: torch.dtype = torch.float32):
        self.d = d
        self.dtype = dtype                 # float32, or bfloat16 / float16: the LayerNorm result rounded
        self.rows = 0                      # total rows appended (device part + spilled part)
        self._dev_rows = 0
        self._max = max_device_rows
        if max_device_rows is not None:
            capacity = min(capacity, max_device_rows)
        self._buf = torch.empty((max(capacity, 1), d), dtype=dtype, device=device)
        self._spilled: list[Tensor] = []

    def _spill(self) -> None:
        if self._dev_rows == 0:
            return
        host = torch.empty((self._dev_rows, self.d), dtype=self.dtype, pin_memory=True)
        host.copy_(self._buf[: self._dev_rows])
        self._spilled.append(host)
        self._dev_rows = 0

    def _reserve(self, extra: int) -> None:
        need = self._dev_rows + extra
        if need <= self._buf.shape[0]:
            return
        if self._max is not None and need > self._max:
            self._spill()
            need = extra
            if need <= self._buf.shape[0]:
                return
        cap = max(need, 2 * self._buf.shape[0])
        if self._max is not None:
            cap = max(need, min(cap, self._max))
        grown = torch.empty((cap, self.d), dtype=self.dtype, device=self._buf.device)
        if self._dev_rows:
            grown[: self._dev_rows].copy_(self._buf[: self._dev_rows])
        self._buf = grown

    def append(self, hidden: Tensor, layer_norm: nn.LayerNorm | None) -> None:
        """Append ``hidden [..., d]`` (flattened), through ``layer_norm`` if given."""
        n = hidden.numel() // self.d
        self._reserve(n)
        lo = self._dev_rows
        if layer_norm is None:
            self._buf[lo:lo + n].copy_(hidden.reshape(n, self.d))
        else:
            ops.layernorm_rows_(hidden, layer_norm.weight.detach(), layer_norm.bias.detach(), layer_norm.eps,
                                self._buf, row0=lo)
        self._dev_rows += n
        self.rows += n

    def tensor(self) -> Tensor:
        """The ``[rows, d]`` matrix: a device view when nothing was spilled, else one host tensor."""
        if not self._spilled:
            return self._buf[: self._dev_rows]
        parts = self._spilled + ([self._buf[: self._dev_rows].cpu()] if self._dev_rows else [])
        return torch.cat(parts, dim=0)


def _hidden_of(output) -> Tensor:
    """Layer output -> hidden states: tuple (transformers 4) or bare tensor (transformers 5)."""
    return output[0] if isinstance(output, (tuple, list)) else output


class WhisperActivationExtractor:
    """Forward hooks on Whisper encoder / decoder layers (hooks.py:40-143)."""

    def __init__(self, model, encoder_layers: list[int] | None = None,
                 decoder_layers: list[int] | None = None, apply_layer_norm: bool = True):
        self.model = model
        self.encoder_layers = encoder_layers or []
        self.decoder_layers = decoder_layers or []
        self.apply_layer_norm = apply_layer_norm
        self.cache = ActivationCache()
        self._hooks: list[torch.utils.hooks.RemovableHandle] = []
        self._encoder_layer_norm = model.model.encoder.layer_norm
        self._decoder_layer_norm = model.model.decoder.layer_norm

    def _normalised(self, hidden: Tensor, layer_norm: nn.LayerNorm) -> Tensor:
        hidden = hidden.detach()
        if not hidden.is_cuda:
            raise RuntimeError("WhisperActivationExtractor (whisper_sae_b200) runs on CUDA models only; "
                               "move the Whisper model and its inputs to the GPU (no CPU fallback)")
        if not self.apply_layer_norm:
            return hidden
        out = torch.empty(hidden.shape, dtype=torch.float32, device=hidden.device)
        ops.layernorm_rows_(hidden, layer_norm.weight.detach(), layer_norm.bias.detach(), layer_norm.eps,
                            out.view(-1, hidden.shape[-1]))
        return out

    def _make_encoder_hook(self, layer_idx: int) -> Callable:
        def hook(module: nn.Module, inputs: tuple, output) -> None:
            act = self._normalised(_hidden_of(output), self._encoder_layer_norm)
            self.cache.encoder.setdefault(layer_idx, []).append(act)
        return hook

    def _make_decoder_hook(self, layer_idx: int) -> Callable:
        def hook(module: nn.Module, inputs: tuple, output) -> None:
            act = self._normalised(_hidden_of(output), self._decoder_layer_norm)
            self.cache.decoder.setdefault(layer_idx, []).append(act)
        return hook

    def register_hooks(self) -> None:
        self.remove_hooks()
        for layer_idx in self.encoder_layers:
            layer = self.model.model.encoder.layers[layer_idx]
            self._hooks.append(layer.register_forward_hook(self._make_encoder_hook(layer_idx)))
        for layer_idx in self.decoder_layers:
            layer = self.model.model.decoder.layers[layer_idx]
            self._hooks.append(layer.register_forward_hook(self._make_decoder_hook(layer_idx)))

    def remove_hooks(self) -> None:
        for h in self._hooks:
            h.remove()
        self._hooks.clear()

    def clear_cache(self) -> None:
        self.cache.clear()

    def __enter__(self) -> "WhisperActivationExtractor":
        self.register_hooks()
        return self

    def __exit__(self, *args) -> None:
        self.remove_hooks()


def run_whisper(model, input_features: Tensor, with_decoder: bool) -> None:
    """Encoder forward, then (optionally) one decoder step from the start token — the forward passes
    hooks.py:181-198 / feature_cache.py:262-279 run while the hooks are registered."""
    encoder_hidden = model.model.encoder(input_features).last_hidden_state
    if with_decoder:
        start = torch.full((input_features.size(0), 1), model.config.decoder_start_token_id,
                           dtype=torch.long, device=input_features.device)
        model.model.decoder(input_ids=start, encoder_hidden_states=encoder_hidden)


def extract_features_batch(model, input_features: Tensor, encoder_layers: list[int],
                           decoder_layers: list[int], apply_layer_norm: bool = True,
                           device: torch.device | str = "cuda") -> dict[str, dict[int, Tensor]]:
    """Activations of one batch (hooks.py:146-210): ``{"encoder": {layer: [B, T, d]}, "decoder": {...}}``,
    fp32 after the final LayerNorm, on ``device``."""
    model.eval()
    input_features = input_features.to(device)
    extractor = WhisperActivationExtractor(model, encoder_layers, decoder_layers, apply_layer_norm)
    with torch.no_grad(), extractor:
        run_whisper(model, input_features, bool(decoder_layers))
    results: dict[str, dict[int, Tensor]] = {"encoder": {}, "decoder": {}}
    for layer_idx in encoder_layers:
        acts = extractor.cache.get_encoder_activations(layer_idx)
        if acts is not None:
            results["encoder"][layer_idx] = acts
    for layer_idx in decoder_layers:
        acts = extractor.cache.get_decoder_activations(layer_idx)
        if acts is not None:
            results["decoder"][layer_idx] = acts
    return results


def flatten_activations(activations: Tensor, component: Literal["encoder", "decoder"]) -> Tensor:
    """``[batch, seq, d] -> [batch * seq, d]`` (hooks.py:213-230)."""
    return activations.reshape(-1, activations.shape[-1])
