"""SAE modules with the reference's public surface, backed by the sm_100a kernels.

Drop-in for ``whisper_sae.sae.model`` (/root/reference/src/whisper_sae/sae/model.py):
``SAEOutput`` (:15-23), ``TopKSAE`` (:26-257), ``ReLUSAE`` (:260-322), ``create_sae`` (:325-354)
keep their signatures, attribute names, parameter/buffer names, shapes, dtypes and
``state_dict`` order.  What changes is *how* ``TopKSAE.forward`` is computed:

* forward  = pack (K0) -> tcgen05 GEMM with fused TopK (K1) -> k-sparse decode + MSE + L0 +
  fired stamps (K2) -> counter bump / dead count (K5); nothing of shape [B, F] is materialised
  unless the caller reads ``output.hidden``;
* backward = sparse K3 (+ tensor-core weight-gradient GEMMs in bf16 mode), returning fp32 grads
  for ``b_pre, encoder.weight, encoder.bias, decoder.weight, decoder.bias``.

Precision: under ``torch.autocast("cuda")`` (what ``SAETrainer`` enables with ``use_amp``) the
encoder GEMM runs in bf16 with fp32 accumulation and the decoder gathers read a bf16 shadow;
otherwise the split-bf16 "fp32-grade" mode is used (see csrc/wsae_pack.cu).  ``precision=`` on the
module overrides the choice.  CUDA only: CPU tensors raise (no CPU fallback by design).

The decoder matrix is stored feature-major (``W_decT[F, d]`` contiguous) so one feature's decoder
vector is one coalesced row; ``decoder.weight`` is exposed as the ``[d, F]`` transposed *view* of
that storage, which keeps ``state_dict`` / optimizer / ``F.normalize(dim=0)`` semantics intact.
"""

from __future__ import annotations

import os
from typing import Callable, Iterator

import torch
from torch import Tensor, nn

from .. import ops
from ..config import SAEConfig

_FIELDS = ("reconstructed", "hidden", "loss", "reconstruction_loss", "sparsity_loss", "l0")


class _LazyOutput:
    """Tuple-like result object whose dense fields may be zero-argument callables: the dense tensors
    are only built when somebody reads them (the trainer never does).  Subclasses set ``_fields``."""

    _fields: tuple[str, ...] = ()
    __slots__ = ("_vals",)

    def __init__(self, *vals, **kw):
        vals = list(vals) + [kw[name] for name in self._fields[len(vals):]]
        if len(vals) != len(self._fields):
            raise TypeError(f"{type(self).__name__} takes {len(self._fields)} fields")
        self._vals = vals

    def _get(self, i: int):
        v = self._vals[i]
        if callable(v) and not isinstance(v, Tensor):
            v = v()
            self._vals[i] = v
        return v

    def __getattr__(self, name: str):
        fields = type(self)._fields
        if name in fields:
            return self._get(fields.index(name))
        raise AttributeError(name)

    def __iter__(self) -> Iterator:
        return (self._get(i) for i in range(len(self._fields)))

    def __len__(self) -> int:
        return len(self._fields)

    def __getitem__(self, i):
        if isinstance(i, slice):
            return tuple(self._get(j) for j in range(len(self._fields))[i])
        return self._get(range(len(self._fields))[i])

    def _asdict(self) -> dict:
        return {name: self._get(i) for i, name in enumerate(self._fields)}

    def __repr__(self) -> str:
        return type(self).__name__ + "(" + ", ".join(self._fields) + ")"


class SAEOutput(_LazyOutput):
    """Result of an SAE forward pass; quacks like the reference's NamedTuple (model.py:15-23):
    ``reconstructed, hidden, loss, reconstruction_loss, sparsity_loss, l0``."""

    _fields = _FIELDS
    __slots__ = ()


_ENCODE_WARNED = False


def _warn_encode_detached() -> None:
    global _ENCODE_WARNED
    if not _ENCODE_WARNED:
        _ENCODE_WARNED = True
        import warnings
        warnings.warn("whisper_sae_b200: encode() returns a tensor without grad_fn (the reference's encode() is "
                      "differentiable); use forward() / output.loss for training, or wrap the call in "
                      "torch.no_grad() to silence this", stacklevel=3)


def _fp32_terms() -> int:
    t = int(os.environ.get("WSAE_FP32_TERMS", "6"))
    if t not in (3, 6):
        raise RuntimeError("WSAE_FP32_TERMS must be 3 or 6")
    return t


_ONES: dict = {}


def _one(device: torch.device) -> Tensor:
    """A resident fp32 scalar 1.0 per device (grad_output of the fused forward pass)."""
    t = _ONES.get(device)
    if t is None:
        t = _ONES[device] = torch.ones((), dtype=torch.float32, device=device)
    return t


class _SparseState:
    """Per-forward sparse results shared between the autograd node and the lazy SAEOutput."""

    __slots__ = ("idx", "val", "resid", "stats", "w_dec_used", "rows_total", "d_out", "mailbox")

    def __init__(self):
        self.idx = self.val = self.resid = self.stats = self.w_dec_used = None
        self.mailbox = None      # graphed train step: the object whose wait_metrics() yields the stats
        self.rows_total = None
        self.d_out = None


class _FusedTopKSAE(torch.autograd.Function):
    """loss = mse(TopK-SAE(x), target) as one autograd node over the fused kernels.

    forward/backward math: model.py:108-148 and its autograd (SURVEY §8 a3-a8).  ``target`` is the
    input itself for an SAE and the MLP output for a transcoder.
    """

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, mod, st: _SparseState, bf16: bool, x, target, b_pre, w_enc, b_enc, w_dec, b_dec):
        same_target = target is None
        tgt = x if same_target else target
        B, d = x.shape
        F = w_enc.shape[0]
        terms = 1 if bf16 else _fp32_terms()
        x = x.contiguous()
        tgt = tgt.contiguous()
        a_packed = ops.pack_activations(x, b_pre, terms)
        w_packed = ops.pack_encoder(w_enc.contiguous(), b_enc, terms)
        idx, val = ops.encode_topk(a_packed, w_packed, B, F, d, terms, mod.k)
        w_decT = w_dec.t()
        if not w_decT.is_contiguous():
            raise RuntimeError("decoder.weight lost its feature-major layout (internal error)")
        w_used = ops.cast_bf16(w_decT) if bf16 else w_decT
        stats = torch.zeros(3, dtype=torch.int64, device=x.device)
        training = bool(mod.training) and getattr(mod, "feature_last_activated", None) is not None
        rows_total = getattr(mod, "_global_rows", None) or B
        d_out = tgt.shape[1]
        # K23 (one pass over the gathered decoder rows for decode + MSE + dv + bias gradients) when a
        # backward will follow: its dv / bias gradients are linear in grad_output, so they are computed
        # here for grad_output = 1 and scaled in backward()
        ctx.fused23 = None
        if (bf16 and any(ctx.needs_input_grad[3:]) and ops.decode_backward_supported(d_out, mod.k, True)
                and ops.wgrad_gemm_supported(d) and ops.wgrad_gemm_supported(d_out)):
            resid = torch.empty((B, d_out), dtype=torch.float32, device=x.device)
            resid_bf = torch.empty((B, d_out), dtype=torch.bfloat16, device=x.device)
            d_b_enc = torch.zeros(F, dtype=torch.float32, device=x.device)
            d_b_dec = torch.zeros(d_out, dtype=torch.float32, device=x.device)
            dpre = torch.empty((B, mod.k), dtype=torch.float32, device=x.device)
            ops.decode_backward(tgt, w_used, b_dec, b_pre, idx, val, _one(x.device),
                                2.0 / (float(rows_total) * float(d_out)),
                                resid=resid, resid_bf16=resid_bf, stats=stats,
                                last_activated=mod.feature_last_activated if training else None,
                                step_count=mod.step_count if training else None,
                                d_b_enc=d_b_enc, d_b_dec=d_b_dec, dpre_val=dpre)
            ctx.fused23 = (resid_bf, d_b_enc, d_b_dec, dpre)
        else:
            resid, _ = ops.decode_mse(
                tgt, w_used, b_dec, b_pre, idx, val, stats=stats,
                last_activated=mod.feature_last_activated if training else None,
                step_count=mod.step_count if training else None,
            )
        if training:
            ops.counters_update(mod.feature_last_activated, mod.step_count,
                                mod.dead_feature_threshold, True, stats[2:])
        numel = float(rows_total) * float(d_out)
        loss = (stats[:1].view(torch.float64)[0] / numel).to(torch.float32)
        st.idx, st.val, st.resid, st.stats, st.w_dec_used, st.rows_total = idx, val, resid, stats, w_used, rows_total
        st.d_out = tgt.shape[1]
        ctx.st = st
        ctx.same_target = same_target
        ctx.bf16 = bf16
        ctx.a_packed = a_packed if bf16 else None   # bf16(x - b_pre): dense operand of the dW_enc GEMM
        ctx.save_for_backward(x, b_pre, w_enc)
        return loss

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, grad_loss):
        st: _SparseState = ctx.st
        x, b_pre, w_enc = ctx.saved_tensors
        needs = ctx.needs_input_grad  # (mod, st, bf16, x, target, b_pre, w_enc, b_enc, w_dec, b_dec)
        B, d_in = x.shape
        F = w_enc.shape[0]
        d_out = st.resid.shape[1]
        dev = x.device
        go = grad_loss.detach().to(torch.float32).contiguous()
        coef = 2.0 / (float(st.rows_total) * float(d_out))
        d_w_enc = torch.zeros((F, d_in), dtype=torch.float32, device=dev) if needs[6] else None
        d_w_decT = torch.zeros((F, d_out), dtype=torch.float32, device=dev) if needs[8] else None
        if ctx.fused23 is None:
            d_b_enc = torch.zeros(F, dtype=torch.float32, device=dev)
            d_b_dec = torch.zeros(d_out, dtype=torch.float32, device=dev)
            dpre = torch.empty(st.idx.shape, dtype=torch.float32, device=dev)
        if ctx.fused23 is not None:
            # dv, db_enc, db_dec came out of K23 in forward() for grad_output = 1
            resid_bf, d_b_enc, d_b_dec, dpre = ctx.fused23
            if d_w_enc is not None or d_w_decT is not None:
                buckets = ops.bucket_by_tile(st.idx, st.val, dpre, F)
                if d_w_enc is not None:
                    ops.wgrad_gemm_(d_w_enc, ctx.a_packed, B, d_in, buckets, buckets.dpre, go, 1.0)
                if d_w_decT is not None:
                    ops.wgrad_gemm_(d_w_decT, resid_bf, B, d_out, buckets, buckets.act, go, coef)
            d_b_enc = d_b_enc * go
            d_b_dec = d_b_dec * go
            if needs[3]:
                dpre = dpre * go
        elif (ctx.bf16 and ops.wgrad_gemm_supported(d_in) and ops.wgrad_gemm_supported(d_out)
              and ops.bucket_supported(F, st.idx.shape[1])):
            resid_bf = torch.empty(st.resid.shape, dtype=torch.bfloat16, device=dev)
            ops.backward_sparse(st.resid, None, None, st.w_dec_used, st.idx, st.val, go, coef,
                                d_w_enc=None, d_w_decT=None, d_b_enc=d_b_enc, d_b_dec=d_b_dec,
                                dpre_val=dpre, resid_bf16=resid_bf)
            if d_w_enc is not None or d_w_decT is not None:
                buckets = ops.bucket_by_tile(st.idx, st.val, dpre, F)
                if d_w_enc is not None:      # dpre already carries coef * grad_out
                    ops.wgrad_gemm_(d_w_enc, ctx.a_packed, B, d_in, buckets, buckets.dpre, None, 1.0)
                if d_w_decT is not None:
                    ops.wgrad_gemm_(d_w_decT, resid_bf, B, d_out, buckets, buckets.act, go, coef)
        elif d_in != d_out and d_w_enc is not None:
            # K3 walks x and the residual with one row width: split off the encoder-gradient scatter
            ops.backward_sparse(st.resid, None, None, st.w_dec_used, st.idx, st.val, go, coef,
                                d_w_enc=None, d_w_decT=d_w_decT, d_b_enc=d_b_enc, d_b_dec=d_b_dec,
                                dpre_val=dpre)
            ops.scatter_rows_(d_w_enc, x, b_pre, st.idx, dpre)
        else:
            ops.backward_sparse(st.resid, x, b_pre, st.w_dec_used, st.idx, st.val, go, coef,
                                d_w_enc=d_w_enc, d_w_decT=d_w_decT, d_b_enc=d_b_enc, d_b_dec=d_b_dec,
                                dpre_val=dpre)
        d_b_pre = None
        if b_pre is not None and needs[5]:
            if ctx.same_target:
                d_b_pre = ops.bpre_grad(d_b_dec, d_b_enc, w_enc)
            else:  # separate target: b_pre only enters through the encoder
                d_b_pre = ops.bpre_grad(torch.zeros(d_in, dtype=torch.float32, device=dev),
                                        d_b_enc, w_enc)
        dx = dtarget = None
        if needs[3]:
            dx = ops.input_grad(st.resid, w_enc, st.idx, dpre, go, coef, subtract_g=ctx.same_target)
        if needs[4] and not ctx.same_target:
            dtarget = st.resid * (-coef * go)
        return (None, None, None, dx, dtarget, d_b_pre, d_w_enc,
                d_b_enc if needs[7] else None,
                d_w_decT.t() if d_w_decT is not None else None,
                d_b_dec if needs[9] else None)


def _feature_major_(linear: nn.Linear) -> None:
    """Re-point ``linear.weight`` ([out=d, in=F]) at feature-major storage: strides (1, d)."""
    w = linear.weight
    d = w.shape[0]
    if w.dim() == 2 and w.stride() == (1, d) and w.data.t().is_contiguous():
        return
    w.data = w.data.t().contiguous().t()


class TopKSAE(nn.Module):
    """TopK sparse autoencoder (reference: model.py:26-257), fused sm_100a implementation."""

    def __init__(
        self,
        input_dim: int,
        hidden_dim: int,
        k: int = 32,
        normalize_decoder: bool = True,
        dead_feature_threshold: int = 10_000,
        precision: str | None = None,
    ):
        super().__init__()
        self.input_dim = input_dim
        self.hidden_dim = hidden_dim
        self.k = k
        self.normalize_decoder = normalize_decoder
        self.dead_feature_threshold = dead_feature_threshold
        if precision not in (None, "bf16", "fp32"):
            raise ValueError("precision must be None, 'bf16' or 'fp32'")
        self.precision = precision

        # Same construction order as the reference so a given torch seed yields the same weights.
        self.encoder = nn.Linear(input_dim, hidden_dim, bias=True)
        self.decoder = nn.Linear(hidden_dim, input_dim, bias=True)
        self.b_pre = nn.Parameter(torch.zeros(input_dim))
        self._init_decoder()
        self.register_buffer("feature_last_activated", torch.zeros(hidden_dim, dtype=torch.long))
        self.register_buffer("step_count", torch.tensor(0, dtype=torch.long))
        _feature_major_(self.decoder)
        self._global_rows: int | None = None  # set by the data-parallel trainer (global batch rows)

    # ------------------------------------------------------------------ init / renorm
    def _init_decoder(self) -> None:
        """xavier-uniform, unit-norm columns, then x0.1 (model.py:81-89)."""
        with torch.no_grad():
            nn.init.xavier_uniform_(self.decoder.weight)
            self.decoder.weight.data = nn.functional.normalize(self.decoder.weight.data, dim=0)
            self.decoder.weight.data *= 0.1

    def _w_decT(self) -> Tensor:
        """Contiguous feature-major [F, d] alias of ``decoder.weight`` (re-laid-out if needed)."""
        _feature_major_(self.decoder)
        return self.decoder.weight.data.t()

    def normalize_decoder_weights(self) -> None:
        """Unit-norm decoder columns, in place (model.py:91-96; the flag is ignored there too)."""
        w = self._w_decT()
        if w.is_cuda:
            ops.renorm_decoder_(w, 1e-12)
        else:  # host-side bookkeeping only (e.g. CPU construction in tests): same formula
            with torch.no_grad():
                w.copy_(nn.functional.normalize(w, dim=1))

    # ------------------------------------------------------------------ forward pieces
    def _use_bf16(self) -> bool:
        if self.precision is not None:
            return self.precision == "bf16"
        return torch.is_autocast_enabled("cuda")

    def _check_input(self, x: Tensor) -> Tensor:
        if not x.is_cuda:
            raise RuntimeError(
                "TopKSAE (whisper_sae_b200) runs on CUDA sm_100a only; move the module and the "
                "batch to a B200 (there is no CPU fallback)"
            )
        if x.dim() != 2 or x.shape[1] != self.input_dim:
            raise RuntimeError(f"expected input of shape [batch, {self.input_dim}], got {tuple(x.shape)}")
        return x

    def _sparse_encode(self, x: Tensor) -> tuple[Tensor, Tensor]:
        bf16 = self._use_bf16()
        terms = 1 if bf16 else _fp32_terms()
        x = x.detach().to(torch.float32).contiguous()
        a = ops.pack_activations(x, self.b_pre.detach(), terms)
        w = ops.pack_encoder(self.encoder.weight.detach().contiguous(), self.encoder.bias.detach(), terms)
        return ops.encode_topk(a, w, x.shape[0], self.hidden_dim, self.input_dim, terms, self.k)

    def encode(self, x: Tensor) -> Tensor:
        """Dense [batch, hidden_dim] TopK activations (model.py:98-118).  NOT differentiable (the
        reference's is): the result carries no grad_fn, so a loss built on ``decode(encode(x))`` would
        train the decoder only - a warning says so once; ``forward`` is the differentiable path."""
        x = self._check_input(x)
        if torch.is_grad_enabled() and (x.requires_grad or self.encoder.weight.requires_grad):
            _warn_encode_detached()
        idx, val = self._sparse_encode(x)
        return ops.densify_hidden(idx, val, self.hidden_dim)

    def decode(self, hidden: Tensor) -> Tensor:
        """hidden @ W_dec^T + b_dec + b_pre (model.py:120-129). Dense input => library GEMM."""
        return nn.functional.linear(hidden, self.decoder.weight, self.decoder.bias) + self.b_pre

    def forward(self, x: Tensor) -> SAEOutput:
        x = self._check_input(x)
        bf16 = self._use_bf16()
        self._w_decT()  # make sure the storage is feature-major before the kernels see it
        st = _SparseState()
        loss = _FusedTopKSAE.apply(self, st, bf16, x, None, self.b_pre, self.encoder.weight,
                                   self.encoder.bias, self.decoder.weight, self.decoder.bias)
        B = x.shape[0]
        F = self.hidden_dim
        x32 = x.detach()

        def _recon() -> Tensor:
            return st.resid + x32.to(torch.float32)

        def _hidden() -> Tensor:
            return ops.densify_hidden(st.idx, st.val, F)

        def _l0() -> Tensor:
            return st.stats[1].to(torch.float32) / float(B)

        def _sparsity() -> Tensor:
            return torch.zeros((), dtype=torch.float32, device=x.device)

        out = SAEOutput(_recon, _hidden, loss, loss, _sparsity, _l0)
        self._last_sparse = st
        return out

    # ------------------------------------------------------------------ dead features
    def _update_dead_features(self, hidden: Tensor) -> None:
        """Dense-input variant kept for API parity (model.py:168-181); forward() uses the fused path."""
        if self.training:
            self.step_count += 1
            active = (hidden > 0).any(dim=0)
            self.feature_last_activated[active] = self.step_count

    def get_dead_features(self) -> Tensor:
        return (self.step_count - self.feature_last_activated) > self.dead_feature_threshold

    def get_dead_feature_ratio(self) -> float:
        return self.get_dead_features().float().mean().item()

    def resample_dead_features(self, inputs: Tensor, num_resample: int | None = None) -> int:
        """Re-point dead features at the highest-error inputs (model.py:197-257), on device.

        Same selection and assignment rules as the reference, vectorised: the i-th dead feature
        (ascending index) receives the i-th highest-error input row, L2-normalised.
        """
        dead_idx = torch.where(self.get_dead_features())[0]
        num_dead = int(dead_idx.numel())
        if num_dead == 0:
            return 0
        if num_resample is not None:
            num_dead = min(num_dead, num_resample)
            dead_idx = dead_idx[:num_dead]
        with torch.no_grad():
            out = self.forward(inputs)
            st = self._last_sparse
            errors = (st.resid.to(torch.float32) ** 2).sum(dim=-1)
            del out
            n = min(num_dead, errors.numel())
            _, top = torch.topk(errors, n)
            rows = nn.functional.normalize(inputs[top].to(torch.float32), dim=-1)
            tgt = dead_idx[:n]
            self.encoder.weight.data[tgt] = rows
            self.encoder.bias.data[tgt] = 0.0
            self._w_decT()[tgt] = rows
            self.feature_last_activated[tgt] = self.step_count
        return num_dead


class ReLUSAE(nn.Module):
    """Dense ReLU + L1 SAE (model.py:260-322).  Genuinely dense GEMMs: left to the library."""

    def __init__(self, input_dim: int, hidden_dim: int, sparsity_weight: float = 0.01,
                 normalize_decoder: bool = True):
        super().__init__()
        self.input_dim = input_dim
        self.hidden_dim = hidden_dim
        self.sparsity_weight = sparsity_weight
        self.normalize_decoder = normalize_decoder
        self.encoder = nn.Linear(input_dim, hidden_dim)
        self.decoder = nn.Linear(hidden_dim, input_dim)
        if normalize_decoder:
            self._unit_columns()

    def _unit_columns(self) -> None:
        with torch.no_grad():
            self.decoder.weight.data = nn.functional.normalize(self.decoder.weight.data, dim=0)

    def normalize_decoder_weights(self) -> None:
        if self.normalize_decoder:
            self._unit_columns()

    def forward(self, x: Tensor) -> SAEOutput:
        hidden = torch.relu(self.encoder(x))
        reconstructed = self.decoder(hidden)
        mse = nn.functional.mse_loss(reconstructed, x)
        l1 = hidden.abs().mean()
        l0 = (hidden > 0).float().sum(dim=-1).mean()
        return SAEOutput(reconstructed, hidden, mse + self.sparsity_weight * l1, mse, l1, l0)


def create_sae(config: SAEConfig, input_dim: int) -> nn.Module:
    """Factory (model.py:325-354): TopKSAE iff activation == "topk", else ReLUSAE."""
    hidden_dim = config.get_hidden_dim(input_dim)
    if config.activation == "topk":
        return TopKSAE(input_dim=input_dim, hidden_dim=hidden_dim, k=config.k,
                       normalize_decoder=config.normalize_decoder,
                       dead_feature_threshold=config.dead_feature_threshold)
    return ReLUSAE(input_dim=input_dim, hidden_dim=hidden_dim,
                   normalize_decoder=config.normalize_decoder)
