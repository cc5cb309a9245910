"""Splice trained TopK SAEs into Whisper's forward pass: spliced-in loss, feature ablation and steering.

A *site* is one ``(component, layer)`` pair, hooked where ``WhisperActivationExtractor`` hooks it: the
output of ``model.model.{encoder,decoder}.layers[i]``.  The site's SAE sees what extraction wrote to the
activation cache, ``x = LN(h)`` with that component's final LayerNorm (or ``x = h`` with
``apply_layer_norm=False``), and the hook returns the layer output with ``h`` replaced by ``h'``:

* ``mode="replace"``: ``h' = LN^-1(recon')`` - Whisper continues on the SAE's reconstruction;
* ``mode="error"``: ``h' = h + LN^-1-scale(recon' - recon)`` - the SAE error term is kept, so only the
  intervention changes the stream, and without one the forward is the clean forward bit for bit.

``recon'`` is the reconstruction after the intervention: a per-feature ``gain`` (0 ablates a feature,
> 1 amplifies it; it acts on the features a row selected) and a ``steer`` vector in the SAE's space added
to every row.  Clamping feature f to c on every row is ``gain[f] = 0`` with ``steer += c * W_dec[:, f]``.
include/wsae.h states the arithmetic.

Per forward and site: ``wsae_splice_pack`` (LayerNorm + K1's packed operand, x never written) -> K1
(``ops.encode_topk``, unchanged) -> ``wsae_splice_decode`` (sparse decode + intervention + inverse
LayerNorm + store in the model's dtype, with the statistics accumulated on the device).  Nothing of shape
``[N, F]`` is built and there is no host synchronisation per forward.  CUDA only; inference only (the
spliced output carries no autograd history).  Transcoders and crosscoders are not supported.
"""

from __future__ import annotations

from dataclasses import dataclass
from typing import Callable

import torch
from torch import Tensor, nn

from .. import ops
from .crosscoder import CrossLayerCrosscoder
from .hooks import _hidden_of
from .model import TopKSAE
from .transcoder import _TranscoderBase

Site = tuple[str, int]
_COMPONENTS = ("encoder", "decoder")


@dataclass(frozen=True)
class SpliceStats:
    """What a site's SAE did on the rows spliced since the last ``reset_stats()``.

    ``mse`` and ``fvu`` measure the unmodified reconstruction against ``x``, whatever the intervention;
    ``fvu = sse / (sum x^2 - ||sum x||^2 / rows)``.  ``l0`` is the mean number of positive selected values
    per row, and ``feature_counts[f] / rows`` the density of feature f on this traffic (0: dead here)."""

    rows: int
    mse: float
    fvu: float
    l0: float
    feature_counts: Tensor      # int64 [F], on the host


@dataclass(frozen=True)
class SpliceEval:
    """``evaluate_splice``: teacher-forced cross-entropies and the per-token KL(clean || spliced)."""

    ce_clean: float
    ce_spliced: float
    ce_zero: float
    loss_recovered: float       # (ce_zero - ce_spliced) / (ce_zero - ce_clean)
    kl: float


class _SiteState:
    __slots__ = ("sae", "d", "F", "k", "ln", "gamma", "beta", "eps", "w_packed", "w_decT", "b_dec", "b_pre",
                 "gain", "steer", "stats", "x_sum", "feature_count", "rows")

    def __init__(self, sae: TopKSAE, layer_norm: nn.LayerNorm):
        self.sae = sae
        self.d, self.F, self.k = sae.input_dim, sae.hidden_dim, sae.k
        self.ln = layer_norm
        self.gamma = self.beta = None          # fp32 copies of the LayerNorm's parameters
        self.eps = float(layer_norm.eps)
        self.w_packed = self.w_decT = self.b_dec = self.b_pre = None
        self.gain = self.steer = None
        self.stats = self.x_sum = self.feature_count = None
        self.rows = 0


class WhisperSAESplice:
    """Context manager that splices ``saes`` (``{("encoder" | "decoder", layer): TopKSAE}``) into
    ``model`` (a transformers ``WhisperForConditionalGeneration``) while it is entered.

    The SAEs' parameters and buffers are never written.  Their packed encoder operand and bf16 decoder
    shadow are built once, when the hooks are first registered; call ``refresh()`` after changing an
    SAE's weights."""

    def __init__(self, model, saes: dict[Site, TopKSAE], mode: str = "replace", apply_layer_norm: bool = True,
                 collect_stats: bool = True):
        if mode not in ops.SPLICE_MODES:
            raise ValueError(f"unknown splice mode {mode!r} (one of {sorted(ops.SPLICE_MODES)})")
        if not saes:
            raise ValueError("no sites to splice")
        self.model = model
        self.mode = mode
        self.apply_layer_norm = apply_layer_norm
        self.collect_stats = collect_stats
        self._hooks: list[torch.utils.hooks.RemovableHandle] = []
        self._sites: dict[Site, _SiteState] = {}
        d_model = int(model.config.d_model)
        for site, sae in saes.items():
            comp, layer = self._check_site_name(site)
            if isinstance(sae, (_TranscoderBase, CrossLayerCrosscoder)):
                raise TypeError(f"site {site}: {type(sae).__name__} is not supported by WhisperSAESplice "
                                "(transcoder and crosscoder splices are out of scope); pass a TopKSAE")
            if not isinstance(sae, TopKSAE):
                raise TypeError(f"site {site}: expected a TopKSAE, got {type(sae).__name__}")
            if sae.input_dim != d_model:
                raise ValueError(f"site {site}: the SAE's input_dim {sae.input_dim} != the model's d_model {d_model}")
            if d_model % 8 != 0 or d_model > ops.SPLICE_MAX_D:
                raise ValueError(f"site {site}: the splice kernels need d_model % 8 == 0 and d_model <= "
                                 f"{ops.SPLICE_MAX_D} (got {d_model})")
            ln = getattr(model.model, comp).layer_norm
            if apply_layer_norm and bool((ln.weight.detach() == 0).any()):
                raise ValueError(f"site {site}: the {comp}'s final LayerNorm has a zero weight, so its inverse "
                                 "does not exist (use apply_layer_norm=False if the SAE was trained on raw outputs)")
            self._sites[(comp, layer)] = _SiteState(sae, ln)

    # ------------------------------------------------------------------ sites and operands
    def _check_site_name(self, site) -> Site:
        if not (isinstance(site, tuple) and len(site) == 2 and site[0] in _COMPONENTS
                and isinstance(site[1], int) and not isinstance(site[1], bool)):
            raise ValueError(f"site {site!r} must be ('encoder' | 'decoder', layer index)")
        comp, layer = site
        n = len(getattr(self.model.model, comp).layers)
        if not 0 <= layer < n:
            raise ValueError(f"site {site!r}: the {comp} has layers 0..{n - 1}")
        return comp, layer

    def _site(self, site) -> _SiteState:
        key = self._check_site_name(site)
        if key not in self._sites:
            raise KeyError(f"site {site!r} is not spliced (sites: {sorted(self._sites)})")
        return self._sites[key]

    def _check_cuda(self) -> None:
        for site, s in self._sites.items():
            dev = s.ln.weight.device
            if not s.ln.weight.is_cuda:
                raise RuntimeError("WhisperSAESplice (whisper_sae_b200) runs on CUDA models only; move the Whisper "
                                   "model and its inputs to the GPU (no CPU fallback)")
            p = s.sae.encoder.weight
            if not p.is_cuda or p.device != dev:
                raise RuntimeError(f"site {site}: the SAE must be on the model's device {dev} (it is on {p.device})")

    def refresh(self) -> None:
        """(Re)build every site's packed encoder operand, bf16 decoder shadow and bias copies from the
        SAE's current weights."""
        self._check_cuda()
        with torch.no_grad():
            for s in self._sites.values():
                sae = s.sae
                s.w_packed = ops.pack_encoder(sae.encoder.weight.detach().float().contiguous(),
                                              sae.encoder.bias.detach().float().contiguous(), 1)
                s.w_decT = ops.cast_bf16(sae.decoder.weight.detach().float().t().contiguous())
                s.b_dec = sae.decoder.bias.detach().float().clone()
                s.b_pre = sae.b_pre.detach().float().clone()
                s.gamma = s.ln.weight.detach().float().contiguous()
                s.beta = s.ln.bias.detach().float().contiguous()
                if self.collect_stats and s.stats is None:
                    dev = s.w_decT.device
                    s.stats = torch.zeros(3, dtype=torch.int64, device=dev)
                    s.x_sum = torch.zeros(s.d, dtype=torch.float64, device=dev)
                    s.feature_count = torch.zeros(s.F, dtype=torch.int64, device=dev)

    # ------------------------------------------------------------------ interventions
    def set_intervention(self, site: Site, gain: Tensor | None = None, steer: Tensor | None = None) -> None:
        """Set the site's intervention: ``gain`` float32 [F] (None: all ones), ``steer`` float32 [d] in the
        SAE's (normalised) space (None: zero), both on the SAE's device."""
        s = self._site(site)
        dev = s.sae.encoder.weight.device
        for name, t, n in (("gain", gain, s.F), ("steer", steer, s.d)):
            if t is None:
                continue
            if not isinstance(t, Tensor) or t.dtype != torch.float32 or tuple(t.shape) != (n,):
                raise ValueError(f"site {site}: {name} must be a float32 tensor of shape [{n}]")
            if t.device != dev:
                raise ValueError(f"site {site}: {name} is on {t.device}, the SAE on {dev}")
        s.gain = None if gain is None else gain.detach().contiguous()
        s.steer = None if steer is None else steer.detach().contiguous()

    def clear_interventions(self) -> None:
        for s in self._sites.values():
            s.gain = s.steer = None

    # ------------------------------------------------------------------ statistics
    def stats(self, site: Site) -> SpliceStats:
        """The site's statistics since the last ``reset_stats()`` (one host synchronisation)."""
        s = self._site(site)
        if not self.collect_stats:
            raise RuntimeError("statistics are off (collect_stats=False)")
        if s.stats is None or s.rows == 0:
            return SpliceStats(0, float("nan"), float("nan"), float("nan"), torch.zeros(s.F, dtype=torch.int64))
        blob = torch.cat([s.stats, s.x_sum.view(torch.int64), s.feature_count]).cpu()
        sse, sumsq = blob[:2].view(torch.float64).tolist()
        l0 = int(blob[2])
        x_sum = blob[3:3 + s.d].view(torch.float64)
        rows = s.rows
        denom = sumsq - float((x_sum * x_sum).sum()) / rows
        return SpliceStats(rows, sse / (rows * s.d), sse / denom if denom > 0 else float("nan"), l0 / rows,
                           blob[3 + s.d:].clone())

    def reset_stats(self) -> None:
        for s in self._sites.values():
            s.rows = 0
            for t in (s.stats, s.x_sum, s.feature_count):
                if t is not None:
                    t.zero_()

    # ------------------------------------------------------------------ the hook
    def _splice(self, s: _SiteState, h: Tensor) -> Tensor:
        h = h.detach()
        if h.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            raise RuntimeError(f"unsupported hidden-state dtype {h.dtype} (float32, bfloat16 or float16)")
        if not h.is_cuda:
            raise RuntimeError("WhisperSAESplice runs on CUDA models only (no CPU fallback)")
        h2 = h.reshape(-1, s.d)
        N = h2.shape[0]
        if N == 0:
            return h
        if not h2.is_contiguous() or h2.data_ptr() % 16 != 0:
            h2 = h2.contiguous()
        if self.apply_layer_norm:
            a_packed, row_stats = ops.splice_pack(h2, s.gamma, s.beta, s.eps, s.b_pre)
            gamma, beta = s.gamma, s.beta
        else:
            slot = torch.full((1,), h2.data_ptr(), dtype=torch.int64, device=h2.device)
            a_packed = ops.pack_activations_at(slot, N, s.d, s.b_pre, x_dtype=h2.dtype)
            row_stats = gamma = beta = None
        idx, val = ops.encode_topk(a_packed, s.w_packed, N, s.F, s.d, 1, s.k)
        out = ops.splice_decode(h2, row_stats, gamma, beta, s.w_decT, s.b_dec, s.b_pre, idx, val, mode=self.mode,
                                gain=s.gain, steer=s.steer, stats=s.stats, x_sum=s.x_sum,
                                feature_count=s.feature_count)
        s.rows += N
        return out.view(h.shape)

    def _make_hook(self, s: _SiteState) -> Callable:
        def hook(module: nn.Module, inputs: tuple, output):
            return _with_hidden(output, self._splice(s, _hidden_of(output)))
        return hook

    def register_hooks(self) -> None:
        self.remove_hooks()
        self._check_cuda()
        if any(s.w_packed is None for s in self._sites.values()):
            self.refresh()
        for (comp, layer), s in self._sites.items():
            mod = getattr(self.model.model, comp).layers[layer]
            self._hooks.append(mod.register_forward_hook(self._make_hook(s)))

    def remove_hooks(self) -> None:
        for h in self._hooks:
            h.remove()
        self._hooks.clear()

    @property
    def active(self) -> bool:
        return bool(self._hooks)

    def __enter__(self) -> "WhisperSAESplice":
        self.register_hooks()
        return self

    def __exit__(self, *args) -> None:
        self.remove_hooks()


def _with_hidden(output, hidden: Tensor):
    """The layer's output structure with its hidden states replaced (the output itself is not modified)."""
    if isinstance(output, tuple):
        return (hidden,) + tuple(output[1:])
    if isinstance(output, list):
        return [hidden] + list(output[1:])
    return hidden


def evaluate_splice(model, input_features: Tensor, labels: Tensor, splice: WhisperSAESplice) -> SpliceEval:
    """Teacher-forced ``model(input_features=..., labels=...)`` three times - clean, spliced, and with the
    splice's site outputs replaced by zeros - and the mean per-token KL(clean || spliced) over the positions
    whose label is not -100.  The splice's hooks are in place afterwards iff they were before."""
    was_active = splice.active
    sites = list(splice._sites)
    with torch.no_grad():
        splice.remove_hooks()
        try:
            clean = model(input_features=input_features, labels=labels)
            splice.register_hooks()
            spliced = model(input_features=input_features, labels=labels)
            splice.remove_hooks()
            zero_hooks = [getattr(model.model, comp).layers[layer].register_forward_hook(
                lambda m, i, o: _with_hidden(o, torch.zeros_like(_hidden_of(o)))) for comp, layer in sites]
            try:
                zero = model(input_features=input_features, labels=labels)
            finally:
                for h in zero_hooks:
                    h.remove()
        finally:
            if was_active:
                splice.register_hooks()
        mask = labels != -100
        lp_clean = torch.log_softmax(clean.logits.float(), dim=-1)
        lp_spliced = torch.log_softmax(spliced.logits.float(), dim=-1)
        kl_tok = (lp_clean.exp() * (lp_clean - lp_spliced)).sum(-1)
        kl = float(kl_tok[mask].mean())
    ce_clean, ce_spliced, ce_zero = float(clean.loss), float(spliced.loss), float(zero.loss)
    denom = ce_zero - ce_clean
    return SpliceEval(ce_clean, ce_spliced, ce_zero,
                      (ce_zero - ce_spliced) / denom if denom != 0 else float("nan"), kl)
