"""SAE trainer with the reference's interface (``whisper_sae.sae.training``,
/root/reference/src/whisper_sae/sae/training.py:19-379) over the fused sm_100a train step.

Same constructor, public attributes, ``train_step`` / ``train_epoch`` / ``train`` /
``setup_scheduler`` / checkpoint + metrics file formats.  Differences that are deliberate:

* the five per-step ``.item()`` host syncs (training.py:207-215) become ONE poll of a 32-byte pinned
  host mailbox the counters kernel posts to ({SSE as float64, L0 count, dead count, sequence word});
  the autograd (non-graphed) path reads the same three numbers with one 24-byte ``stats.cpu()``;
* ``use_amp`` selects the bf16 tensor-core path instead of fp16 autocast.  bf16 keeps the fp32
  exponent range, so loss scaling is the identity: ``self.scaler`` is still a ``GradScaler``
  (attribute preserved) but constructed disabled unless ``grad_scaler=True`` is passed; the fused
  autograd node honours an arbitrary scalar ``grad_output`` either way;
* ``fused_optimizer=True`` (default on CUDA) runs clip-by-global-norm + AdamW as one pass per
  parameter over the optimizer's own state tensors (csrc/wsae_elementwise.cu), so
  ``optimizer.state_dict()`` checkpoints stay interchangeable with ``torch.optim.AdamW``.
"""

from __future__ import annotations

import contextlib
import gc
import json
import math
import os
import weakref
from dataclasses import asdict, dataclass
from pathlib import Path

import numpy as np
import torch
from rich.progress import BarColumn, Progress, SpinnerColumn, TaskProgressColumn, TextColumn
from torch import Tensor
from torch.optim import AdamW
from torch.optim.lr_scheduler import CosineAnnealingLR, LinearLR, SequentialLR
from torch.utils.data import DataLoader

from .. import ops
from ..config import TrainingConfig
from ..data.feature_cache import IndexedBatch
from .model import SAEOutput, TopKSAE, _fp32_terms, _SparseState


# largest k the graphed train step (and with it data_parallel=True) serves: K1 runs fused (k <= 64)
# or chunked, K23 up to 256 (ops.decode_backward_supported), the K4 bucketing up to ~265.  Larger k
# trains through the autograd node, eagerly.
GRAPH_MAX_K = 256
# batch dtypes the graphed step trains on (half batches are read in place or staged to fp32, exactly)
_X_DTYPES = (torch.float32, torch.bfloat16, torch.float16)


@dataclass
class TrainingMetrics:
    """Per-step metrics (training.py:19-29)."""

    loss: float
    reconstruction_loss: float
    sparsity_loss: float
    l0: float
    dead_feature_ratio: float
    learning_rate: float
    step: int


def _ensure_adamw_state(optimizer: AdamW, p: Tensor) -> dict:
    """AdamW state for ``p`` exactly as torch.optim.AdamW creates it (float32 CPU ``step``), with the
    moments in the parameter's own dense layout so flat elementwise kernels can walk the storage."""
    st = optimizer.state[p]
    if len(st) == 0:
        st["step"] = torch.tensor(0.0, dtype=torch.float32)
        st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
        st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
    for name in ("exp_avg", "exp_avg_sq"):
        t = st[name]
        if t.stride() != p.stride() or t.device != p.device:
            st[name] = torch.empty_strided(p.shape, p.stride(), dtype=p.dtype, device=p.device).copy_(t)
    return st


@contextlib.contextmanager
def _quiet_gc():
    """Stream capture is invalidated by ANY forbidden CUDA call in the process, and destroying another
    CUDA graph is one: a dead trainer (trainer <-> graphed-step reference cycle) that Python's cyclic
    collector happens to free in the middle of a capture kills it (cudaErrorStreamCaptureInvalidated;
    torch.cuda.graph stopped collecting up front in 2.9).  Collect before, keep the collector off inside."""
    gc.collect()
    was_on = gc.isenabled()
    gc.disable()
    try:
        yield
    finally:
        if was_on:
            gc.enable()


_DP_GRAPH_TRAINERS: "weakref.WeakSet[SAETrainer]" = weakref.WeakSet()


def _guard_process_group_teardown(trainer: "SAETrainer") -> None:
    """Whole-step capture with the NCCL collectives inside (WSAE_DP_GRAPH=1): destroying the communicator
    while a captured graph still holds its kernels blocks forever (what looked like a capture hang in
    round 1 was exactly this, at the end of the run).  Live trainers therefore drop their graphs right
    before ``torch.distributed.destroy_process_group`` and at interpreter exit."""
    import atexit

    import torch.distributed as dist

    _DP_GRAPH_TRAINERS.add(trainer)

    def release_all() -> None:
        for tr in list(_DP_GRAPH_TRAINERS):
            tr.release_graphs()

    if not getattr(dist.destroy_process_group, "_wsae_guard", False):
        original = dist.destroy_process_group

        def destroy_process_group(*args, **kwargs):
            release_all()
            return original(*args, **kwargs)

        destroy_process_group._wsae_guard = True
        dist.destroy_process_group = destroy_process_group
        atexit.register(release_all)


class _GraphedStep:
    """One full train step (K0..K5 + clip + AdamW + renorm) at a fixed batch shape, launched from a
    CUDA graph: the per-step host work drops from ~40 launches to one ``replay()``.

    No autograd: the kernels are called in the same order the autograd node would run them, with
    ``grad_output = 1``.  The first call runs the body eagerly (it is a real step and also warms
    up per-function attributes), the second call captures, later calls replay.  Learning rate and
    Adam bias corrections live in a device ``hyper`` vector refreshed from pinned memory before
    every replay, so the captured graph never goes stale.
    """

    def __init__(self, trainer: "SAETrainer", rows: int):
        m = trainer.model
        dev = m.b_pre.device
        self.trainer = trainer
        self.rows = rows
        self.bf16 = bool(trainer.use_amp)
        # per-step control block, ONE 64-byte H2D copy from pinned memory before every replay:
        # [hyper f32[8] | x_slot i64 | seq i64 | rows_slot i64 | pad].  x_slot holds the device address of the step's batch:
        # the kernels that read the activations (K0 pack, K23 target) take it from there when they
        # RUN, so the captured graph trains on a device-resident batch in place; only batches that
        # arrive on the host (or misaligned / non-contiguous) are staged into `x`.
        self.ctl = torch.zeros(64, dtype=torch.uint8, device=dev)
        self.ctl_host = torch.zeros(64, dtype=torch.uint8).pin_memory()
        self.hyper = self.ctl[:32].view(torch.float32)
        self.hyper_host = self.ctl_host[:32].view(torch.float32)
        self.x_slot = self.ctl[32:40].view(torch.int64)
        self.x_slot_host = self.ctl_host[32:40].view(torch.int64)
        # seq numbers the steps; the counters kernel posts {sse, l0, dead, seq} to a pinned mailbox as
        # soon as the metrics are final and SAETrainer._read_metrics polls the sequence word instead
        # of synchronising with the stream (the reference's five `.item()` calls, training.py:206-214)
        self.seq_dev = self.ctl[40:48].view(torch.int64)
        self.seq_host = self.ctl_host[40:48].view(torch.int64)
        # rows_slot: address of an int64 row-index array (0 = identity): an IndexedBatch of a resident
        # activation matrix is gathered INSIDE K0 / K23 (wsae_*_rows_at), never materialised
        self.rows_slot = self.ctl[48:56].view(torch.int64)
        self.rows_slot_np = self.ctl_host[48:56].view(torch.int64).numpy()
        self.mailbox = torch.zeros(4, dtype=torch.int64).pin_memory()
        self.mailbox_np = self.mailbox.numpy()
        self.seq = 0
        # numpy views of the pinned control block: a torch index-assignment costs ~5 us each on the
        # host, which is the critical path once the GPU no longer waits for a stream sync (B = 128)
        self.hyper_np = self.hyper_host.numpy()
        self.x_slot_np = self.x_slot_host.numpy()
        self.seq_np = self.seq_host.numpy()
        self._step_views: list = []       # (optimizer `step` tensor, its 0-d numpy view) per parameter
        d_in, k_sel = m.input_dim, m.k
        # the deterministic step takes K23 wherever its deterministic form exists (33 <= k <= 64 included),
        # so staging and the K23 / K2 + K3 choice in _compute_a follow the same predicate
        self.in_place = (self.bf16 and d_in % 8 == 0 and ops.wgrad_gemm_supported(d_in)
                         and ops.decode_backward_supported(d_in, k_sel, True, bool(trainer.deterministic)))
        # Single-GPU bf16 step: the small kernels that do not sit on the K0 -> K1 -> K23 -> K4 chain run
        # on a side stream (a forked branch of the captured graph): [encoder pack, decoder bf16 cast]
        # next to the activation pack, and [counters + mailbox, b_pre gradient] next to the bucketing
        # and the two weight-gradient GEMMs.  Their outputs are pre-allocated, so no allocation ever
        # changes streams.  0.7945 -> 0.7799 ms per step (same-box A/B); WSAE_FORK=0 switches it off.
        self.fork = os.environ.get("WSAE_FORK", "1") != "0" and not trainer.data_parallel and self.bf16
        self._side = torch.cuda.Stream(device=dev) if self.fork else None
        # small batches: the two weight-gradient GEMMs (24 feature tiles x a few row chunks each at the
        # YAML batch) leave most SMs idle, so dW_dec runs beside dW_enc on a second branch of the graph
        # (96.9 -> 92.7 us per step at 128 rows; no gain from 1024 rows on: profiles/r2c_k4_fork_ab.txt)
        self.fork_k4 = self.fork and rows <= int(os.environ.get("WSAE_FORK_K4_ROWS", "512"))
        # batches of a few hundred rows (the shipped YAML batch is 128): one block per row does the TopK
        # selection, K23 and both weight-gradient rows in ONE launch (wsae_row_step.cu) instead of the
        # five dependent launches rowwise top-k -> K23 -> bucketing -> 2 x K4
        self.row_step = (self.in_place and not trainer.data_parallel and not trainer.deterministic
                         and ops.row_step_supported(rows, d_in, m.hidden_dim, k_sel, True))
        self._side2 = torch.cuda.Stream(device=dev) if self.fork_k4 else None
        self._k4_forked = False
        self._w_packed_buf: Tensor | None = None
        self._w_used_buf: Tensor | None = None
        self._x: Tensor | None = None     # staging buffer, allocated on first use
        # Half-precision batches: the kernels that read the batch through x_slot (K0, K23, the row step)
        # convert each element to fp32 as they load it, and their element type is baked into the captured
        # graph.  So there is one captured graph per dtype the slot has named: `graph` / `_exec` /
        # `kernels_per_replay` belong to the current `x_dtype`, the others wait in `_captured`.  Routes
        # that do not read through the slot stage every batch into the fp32 `x` (an exact conversion).
        self.x_dtype = torch.float32
        self._captured: dict = {}         # dtype -> (graph, exec handle, kernels_per_replay)
        self._warm: set = set()           # dtypes whose step has run eagerly once (loads their kernels)
        self._xh: dict = {}               # per half dtype: staging buffer of host batches on in-place routes
        self.captures = 0
        self._live: Tensor | None = None  # the batch the slot names (kept alive until the next step)
        self.one = torch.ones((), dtype=torch.float32, device=dev)
        self.params = [m.b_pre, m.encoder.weight, m.encoder.bias, m.decoder.weight, m.decoder.bias]
        m._w_decT()
        F, d = m.hidden_dim, m.input_dim
        # one flat gradient bucket (segments 64-byte aligned): a single memset and a single
        # sum-of-squares pass per step; also the unit a data-parallel all-reduce ships
        # layout [b_pre | b_enc | b_dec | W_enc | W_decT]: the three small tensors are one contiguous piece
        sizes = [d, F, d, F * d, F * d]
        starts, off = [], 0
        for n in sizes:
            starts.append(off)
            off += (n + 15) // 16 * 16
        # the step's accumulators share one allocation so ONE memset per step clears them all:
        # [gradient bucket | stats int64[3] | grad sum-of-squares f64] (tail 64-byte aligned)
        self.zeroed = torch.zeros(off + 16, dtype=torch.float32, device=dev)
        self.g_flat = self.zeroed[:off]
        tail = self.zeroed[off:off + 16].view(torch.int64)
        self.stats = tail[0:3]
        self.sumsq = tail[3:4].view(torch.float64)
        self.ticket = tail[4:5]           # block-completion ticket of the row step (zeroed with the rest)
        seg = [self.g_flat[s0:s0 + n] for s0, n in zip(starts, sizes)]
        self.g_b_pre, self.g_b_enc, self.g_b_dec = seg[0], seg[1], seg[2]
        self.g_w_enc, self.g_w_decT = seg[3].view(F, d), seg[4].view(F, d)
        # data-parallel exchange in three contiguous pieces: dW_enc starts as soon as its GEMM is
        # done and overlaps the dW_dec GEMM; the small tensors and W_decT follow
        self.g_part_w_enc = self.g_flat[starts[3]:starts[4]]
        self.g_part_head = self.g_flat[:starts[3]]
        self.g_part_tail = self.g_flat[starts[4]:]
        # sharded optimizer (sae/parallel.py): reduce-scatter the two weight-gradient matrices by
        # feature rows, clip + AdamW + renorm on this rank's rows only, all-gather the updated rows
        comm = trainer.dp_comm
        self.shard = bool(trainer.data_parallel and trainer.shard_optimizer and comm is not None
                          and comm.world > 1 and F % comm.world == 0 and not trainer.deterministic)
        self.f0, self.f1 = comm.row_block(F) if self.shard else (0, F)
        # bf16 operand gather (sharded optimizer, bf16 step): after its AdamW pass a rank packs / casts
        # only ITS updated rows into the bf16 operands K1 and K23 read (W' and the decoder shadow) and
        # those rows are all-gathered - half the bytes of gathering the fp32 weights, and the encoder
        # pack / decoder cast passes shrink by 1/N.  The fp32 rows other ranks own go stale in this
        # replica until SAETrainer.consolidate_weights() gathers them (checkpoints, resampling, epoch end).
        self.zero = bool(self.shard and self.bf16 and os.environ.get("WSAE_DP_OPERANDS", "1") != "0")
        self._zeros_d: Tensor | None = None
        self._early = None
        self.grads = [self.g_b_pre, self.g_w_enc, self.g_b_enc, self.g_w_decT, self.g_b_dec]
        # what autograd would leave in .grad (decoder.weight's grad is the [d, F] transposed view)
        self._grad_views = [g.t() if p is m.decoder.weight else g for p, g in zip(self.params, self.grads)]
        self.state = _SparseState()
        # deterministic mode workspaces (bf16 step with K23 + K4 only)
        self.det = bool(trainer.deterministic) and self.bf16 and ops.wgrad_gemm_supported(d_in) \
            and ops.decode_backward_supported(d_in, k_sel, True, deterministic=True)
        if trainer.deterministic and not self.det:
            raise RuntimeError("deterministic=True covers the bf16 (use_amp) graphed step with d % 8 == 0 and "
                               "k <= 32, or d % 128 == 0 and k <= 256")
        self.det_k23 = self.det_k4 = self.det_sumsq = self.det_bpre = None
        if self.det:
            self.det_k23 = torch.zeros(F + d + 1, dtype=torch.int64, device=dev)
            ws_bytes = ops.wgrad_gemm_workspace(rows, F, d)
            self.det_k4 = torch.empty(max(ws_bytes // 4, 1), dtype=torch.float32, device=dev) if ws_bytes else None
            self.det_sumsq = torch.empty(1024, dtype=torch.float64, device=dev)
            self.det_bpre = torch.empty((F + 255) // 256 * d, dtype=torch.float32, device=dev)
        self.graph: torch.cuda.CUDAGraph | list | None = None
        self._exec: int | list | None = None     # cudaGraphExec_t of `graph` / of its segments (raw launch, see _launch_graph)
        self._mid: dict = {}
        self.kernels_per_replay = 0
        self.calls = 0
        for p in self.params:
            _ensure_adamw_state(trainer.optimizer, p)
        self._ptrs: tuple[int, ...] = ()

    @property
    def x(self) -> Tensor:
        if self._x is None:
            m = self.trainer.model
            self._x = torch.empty((self.rows, m.input_dim), dtype=torch.float32, device=m.b_pre.device)
        return self._x

    def _pointer_key(self) -> tuple[int, ...]:
        m = self.trainer.model
        opt_state = self.trainer.optimizer.state
        # the AdamW moments are not in the per-step key: optimizer.load_state_dict replaces them together with
        # the `step` tensors, which run() notices (and then drops the graph) when it validates its step views
        ptrs = [p.data_ptr() for p in self.params]
        ptrs += [m.feature_last_activated.data_ptr(), m.step_count.data_ptr()]
        return tuple(ptrs)

    def _body(self) -> None:
        self._compute()
        if self.trainer.data_parallel:      # batch-sharded: exchange gradients / stats / fired stamps
            self._exchange()
        self._update_pre()
        if self.shard:
            self.trainer.dp_comm.all_reduce_sum(self.sumsq)
        self._update_opt()
        if self.shard:
            self._gather_weights()

    def _operands(self) -> tuple[Tensor, Tensor]:
        """The trainer-wide bf16 operand buffers of the operand-gather mode (shared by every batch shape)."""
        tr = self.trainer
        if tr._dp_operands is None:
            m = tr.model
            F, d = m.hidden_dim, m.input_dim
            ps = ops.packed_shape(d, 1)
            dev = m.b_pre.device
            tr._dp_operands = (torch.empty(((F + 255) // 256 * 256, ps.kp), dtype=torch.bfloat16, device=dev),
                               torch.empty((F, d), dtype=torch.bfloat16, device=dev))
            tr._dp_operands_fresh = False
        return tr._dp_operands

    def _refresh_operands(self) -> None:
        """Full local pack / cast from the fp32 weights (first step, after consolidate_weights / a load)."""
        m = self.trainer.model
        w_packed, w_used = self._operands()
        ops.pack_encoder(m.encoder.weight.data, m.encoder.bias.data, 1, out=w_packed)
        ops.cast_bf16(m.decoder.weight.data.t(), out=w_used)
        self.trainer._dp_operands_fresh = True

    def _exchange(self) -> None:
        """The per-step collectives behind the kernels (gradients, {sse, l0}, fired stamps)."""
        comm = self.trainer.dp_comm
        last = self.trainer.model.feature_last_activated
        if self.shard:
            h_enc = self._early if self._early is not None else comm.reduce_scatter_rows_async(self.g_w_enc)
            h_dec = comm.reduce_scatter_rows_async(self.g_w_decT)
            comm.all_reduce_sum(self.g_part_head)
            if self.zero:
                # db_pre = db_dec - db_enc . W_enc needs every fp32 encoder row, and this replica only keeps
                # its own rows current: GEMV over those rows with the SUMMED db_enc, then a d-float all-reduce
                m = self.trainer.model
                if self._zeros_d is None:
                    self._zeros_d = torch.zeros_like(self.g_b_dec)
                ops.bpre_grad(self.g_b_dec if comm.rank == 0 else self._zeros_d, self.g_b_enc[self.f0:self.f1],
                              m.encoder.weight.data[self.f0:self.f1], out=self.g_b_pre)
                comm.all_reduce_sum(self.g_b_pre)
            comm.reduce_stats(self.stats, last)
            h_enc.wait()
            h_dec.wait()
        else:
            parts = [self.g_part_head, self.g_part_tail] if self._early is not None else [self.g_flat]
            comm.reduce_step(parts, self.stats, last)
            if self._early is not None:
                self._early.wait()
        self._early = None

    def _start_early(self) -> None:
        """dW_enc is final after its GEMM: start its exchange while the dW_dec GEMM runs."""
        comm = self.trainer.dp_comm
        self._early = (comm.reduce_scatter_rows_async(self.g_w_enc) if self.shard
                       else comm.all_reduce_sum_async(self.g_part_w_enc))

    def _gather_weights(self) -> None:
        m = self.trainer.model
        comm = self.trainer.dp_comm
        if self.zero:
            F = m.hidden_dim
            f0, f1 = self.f0, self.f1
            w_packed, w_used = self._operands()
            ops.pack_encoder_rows_(m.encoder.weight.data[f0:f1], m.encoder.bias.data[f0:f1], 1, w_packed[f0:f1])
            ops.cast_bf16(m.decoder.weight.data.t()[f0:f1], out=w_used[f0:f1])
            comm.all_gather_rows(w_packed[:F])
            comm.all_gather_rows(w_used)
            return
        comm.all_gather_rows(m.encoder.weight.data)
        comm.all_gather_rows(m.decoder.weight.data.t())     # feature-major storage: [F, d] contiguous

    def _compute(self) -> None:
        """Forward + backward kernels of this rank's rows: fills g_flat, stats[0:2], fired stamps."""
        self._compute_a()
        if self._mid["use_gemm"] and self.trainer.data_parallel:   # exchange dW_enc while the dW_dec GEMM runs
            self._start_early()
        self._compute_b()

    def _compute_a(self) -> None:
        """Up to and including the dW_enc GEMM (everything the early all-reduce of dW_enc waits for)."""
        m = self.trainer.model
        B, d = self.rows, m.input_dim
        x = None if self.in_place else self.x      # in place: the kernels read the batch through x_slot
        dev = m.b_pre.device
        F, k = m.hidden_dim, m.k
        terms = 1 if self.bf16 else _fp32_terms()
        w_decT = m.decoder.weight.data.t()
        self.zeroed.zero_()
        if self.det:
            self.det_k23.zero_()
        main = torch.cuda.current_stream()
        if self.fork:
            if self._w_used_buf is None:
                self._w_used_buf = torch.empty((F, d), dtype=torch.bfloat16, device=dev)
            self._side.wait_stream(main)
            with torch.cuda.stream(self._side):
                w_packed = self._w_packed_buf = ops.pack_encoder(
                    m.encoder.weight.data, m.encoder.bias.data, terms, out=self._w_packed_buf)
                if self._side2 is None:
                    w_used = ops.cast_bf16(w_decT, out=self._w_used_buf)
            if self._side2 is not None:      # small batches: the two weight-side kernels side by side
                self._side2.wait_stream(main)
                with torch.cuda.stream(self._side2):
                    w_used = ops.cast_bf16(w_decT, out=self._w_used_buf)
        if self.in_place:
            a_packed = ops.pack_activations_at(self.x_slot, B, d, m.b_pre.data, rows_at=self.rows_slot,
                                               x_dtype=self.x_dtype)
        else:
            a_packed = ops.pack_activations(x, m.b_pre.data, terms)
        if self.fork:
            main.wait_stream(self._side)
            if self._side2 is not None:
                main.wait_stream(self._side2)
        elif self.zero:
            w_packed, w_used = self._operands()      # gathered at the end of the previous step
        else:
            w_packed = ops.pack_encoder(m.encoder.weight.data, m.encoder.bias.data, terms)
        rows_total = m._global_rows or B
        coef = 2.0 / (float(rows_total) * d)
        if self.row_step:
            if not self.fork:
                w_used = ops.cast_bf16(w_decT)
            pre = ops.encode_dense(a_packed, w_packed, B, F, d, terms)
            idx, val = ops.row_step(pre, self.x_slot, w_used, m.decoder.bias.data, m.b_pre.data, self.one, coef, k,
                                    stats=self.stats, last_activated=m.feature_last_activated,
                                    step_count=m.step_count, d_b_enc=self.g_b_enc, d_b_dec=self.g_b_dec,
                                    d_w_enc=self.g_w_enc, d_w_decT=self.g_w_decT, target_is_slot=True,
                                    rows_at=self.rows_slot, w_enc=m.encoder.weight.data, d_b_pre=self.g_b_pre,
                                    finish=(self.ticket, m.dead_feature_threshold, self.stats[2:], self.seq_dev,
                                            self.mailbox),      # counters + metrics mailbox by the last block
                                    x_dtype=self.x_dtype)
            self._k4_forked = False
            self._mid = dict(use_gemm=False, buckets=None, resid_bf=None, B=B, d=d, coef=coef)
            st = self.state
            st.idx, st.val, st.resid, st.stats, st.w_dec_used, st.rows_total = idx, val, None, self.stats, w_used, rows_total
            st.d_out = d
            return
        idx, val = ops.encode_topk(a_packed, w_packed, B, F, d, terms, k)
        if not self.fork and not self.zero:
            w_used = ops.cast_bf16(w_decT) if self.bf16 else w_decT
        dpre = torch.empty((B, k), dtype=torch.float32, device=dev)
        use_gemm = self.bf16 and ops.wgrad_gemm_supported(d)
        if use_gemm and ops.decode_backward_supported(d, k, True, self.det):
            # K23: decode + MSE + stamps + dv + bias gradients in one pass over the gathered rows
            resid = None          # fp32 residual only on demand (SAEOutput.reconstructed, resampling)
            resid_bf = torch.empty((B, d), dtype=torch.bfloat16, device=dev)
            ops.decode_backward(self.x_slot if self.in_place else x, w_used, m.decoder.bias.data,
                                m.b_pre.data, idx, val, self.one, coef,
                                resid=None, resid_bf16=resid_bf, stats=self.stats,
                                last_activated=m.feature_last_activated, step_count=m.step_count,
                                d_b_enc=self.g_b_enc, d_b_dec=self.g_b_dec, dpre_val=dpre,
                                target_is_slot=self.in_place,
                                rows_at=self.rows_slot if self.in_place else None, det_ws=self.det_k23,
                                x_dtype=self.x_dtype)
        else:
            resid, _ = ops.decode_mse(x, w_used, m.decoder.bias.data, m.b_pre.data, idx, val,
                                      stats=self.stats, last_activated=m.feature_last_activated,
                                      step_count=m.step_count)
            if use_gemm:
                resid_bf = torch.empty((B, d), dtype=torch.bfloat16, device=dev)
                ops.backward_sparse(resid, None, None, w_used, idx, val, self.one, coef, d_w_enc=None,
                                    d_w_decT=None, d_b_enc=self.g_b_enc, d_b_dec=self.g_b_dec,
                                    dpre_val=dpre, resid_bf16=resid_bf)
            else:
                ops.backward_sparse(resid, x, m.b_pre.data, w_used, idx, val, self.one, coef,
                                    d_w_enc=self.g_w_enc, d_w_decT=self.g_w_decT,
                                    d_b_enc=self.g_b_enc, d_b_dec=self.g_b_dec, dpre_val=dpre)
        if self.fork:
            self._side.wait_stream(main)
            with torch.cuda.stream(self._side):      # joined in _update, before the gradient norm
                self._counters()
                ops.bpre_grad(self.g_b_dec, self.g_b_enc, m.encoder.weight.data, out=self.g_b_pre,
                              det_ws=self.det_bpre)
        elif not self.trainer.data_parallel:
            # the metrics are final once K23 has run: post them now, so the host has them (and the
            # next step queued) long before the weight-gradient GEMMs and the optimizer finish
            self._counters()
        buckets = None
        if use_gemm:
            # weight gradients on the tensor cores (K4)
            buckets = ops.bucket_by_tile(idx, val, dpre, F)
            self._k4_forked = self.fork_k4 and not self.det     # (the ordered split-K workspace is shared)
            if self._k4_forked:
                self._side2.wait_stream(main)
                with torch.cuda.stream(self._side2):     # joined in _update_pre, before the gradient norm
                    ops.wgrad_gemm_(self.g_w_decT, resid_bf, B, d, buckets, buckets.act, self.one, coef)
            ops.wgrad_gemm_(self.g_w_enc, a_packed, B, d, buckets, buckets.dpre, None, 1.0,
                            det_ws=self.det_k4 if self.det else None)
        else:
            resid_bf = None
        self._mid = dict(use_gemm=use_gemm, buckets=buckets, resid_bf=resid_bf, B=B, d=d, coef=coef)
        s = self.state
        s.idx, s.val, s.resid, s.stats, s.w_dec_used, s.rows_total = idx, val, resid, self.stats, w_used, rows_total
        s.d_out = d

    def _compute_b(self) -> None:
        """The dW_dec GEMM and the b_pre gradient."""
        m = self.trainer.model
        mid = self._mid
        if mid["use_gemm"] and not self._k4_forked:
            ops.wgrad_gemm_(self.g_w_decT, mid["resid_bf"], mid["B"], mid["d"], mid["buckets"],
                            mid["buckets"].act, self.one, mid["coef"],
                            det_ws=self.det_k4 if self.det else None)
        if not self.fork and not self.zero and not self.row_step:   # operand-gather mode: after the exchange
            ops.bpre_grad(self.g_b_dec, self.g_b_enc, m.encoder.weight.data, out=self.g_b_pre,
                          det_ws=self.det_bpre)

    def _update_pre(self) -> None:
        """Counters and the gradient sum of squares on the (possibly reduced) gradient bucket."""
        if self.trainer.data_parallel:      # needs the all-reduced stats / fired stamps
            self._counters()
        if self.fork:
            torch.cuda.current_stream().wait_stream(self._side)
        if self._k4_forked:
            torch.cuda.current_stream().wait_stream(self._side2)
        if self.shard:
            # this rank's rows of the two matrices; the (all-reduced) small tensors count once
            ops.sumsq_(self.g_w_enc[self.f0:self.f1], self.sumsq)
            ops.sumsq_(self.g_w_decT[self.f0:self.f1], self.sumsq)
            if self.trainer.dp_comm.rank == 0:
                ops.sumsq_(self.g_part_head, self.sumsq)
        else:
            ops.sumsq_(self.g_flat, self.sumsq, det_ws=self.det_sumsq)

    def _update_opt(self) -> None:
        """Clip + AdamW + decoder renorm (sharded: on this rank's feature rows and the small tensors)."""
        m = self.trainer.model
        d = m.input_dim
        opt_state = self.trainer.optimizer.state
        entries = []
        for p, g in zip(self.params, self.grads):
            st = opt_state[p]
            is_dec = p is m.decoder.weight          # feature-major storage: rows = decoder vectors
            flags = ops.ADAMW_PROJECT_GRAD if (is_dec and self.trainer.project_decoder_grad) else 0
            pd, ea, es = p.data, st["exp_avg"], st["exp_avg_sq"]
            if self.shard and p.dim() == 2:
                if is_dec:
                    pd, ea, es = pd.t(), ea.t(), es.t()
                pd, g, ea, es = (t[self.f0:self.f1] for t in (pd, g, ea, es))
            entries.append((pd, g, ea, es, d if is_dec else 0, flags))
        ops.adamw_multi_(entries, self.hyper, self.sumsq, 1e-12)   # clip + AdamW + decoder renorm

    def _counters(self) -> None:
        m = self.trainer.model
        ops.counters_update(m.feature_last_activated, m.step_count, m.dead_feature_threshold, True,
                            self.stats[2:], post=(self.stats[:2], self.seq_dev, self.mailbox))

    def _launch_graph(self) -> None:
        """cudaGraphLaunch of the captured step on the current stream.  torch's CUDAGraph.replay() costs
        ~25 us of host time per call (generator bookkeeping, guards); the YAML-batch step's GPU floor is
        ~60 us, so the raw launch through the library (wsae_graph_launch) keeps the loop GPU-bound."""
        if self._exec is None:
            self._exec = self._raw_exec(self.graph)
        self._launch_one(self.graph, self._exec)

    @staticmethod
    def _raw_exec(graph: torch.cuda.CUDAGraph) -> int:
        raw = getattr(graph, "raw_cuda_graph_exec", None)
        if raw is not None and os.environ.get("WSAE_RAW_LAUNCH", "1") != "0":
            try:
                return int(raw())
            except Exception:  # noqa: BLE001 - older torch / not instantiated: CUDAGraph.replay() it is
                return 0
        return 0

    @staticmethod
    def _launch_one(graph: torch.cuda.CUDAGraph, handle: int) -> None:
        if handle:
            ops.graph_launch(handle)
        else:
            graph.replay()

    def wait_metrics(self) -> tuple[float, int, int]:
        """(sse, l0 count, dead count) of the step launched last: polls the mailbox's sequence word."""
        mb, seq = self.mailbox_np, self.seq
        spins = 0
        while mb[3] != seq:
            spins += 1
            if spins > 4_000_000:           # ~1 s: a very long step, or a fault - let CUDA say which
                torch.cuda.synchronize(self.ctl.device)
                if mb[3] != seq:
                    raise RuntimeError("train step finished without posting its metrics")
        return float(mb[:1].view("float64")[0]), int(mb[1]), int(mb[2])

    def run(self, batch: Tensor) -> None:
        """Launch first, book-keep afterwards: everything the GPU needs (batch copy, hyper vector,
        pointer check) is issued before the replay; the optimizer's ``step`` tensors and the grad
        views are updated while the kernels run (matters at the launch-bound YAML batch sizes)."""
        tr = self.trainer
        rows_ptr = 0
        if isinstance(batch, IndexedBatch):
            f, r = batch.features, batch.rows
            if (self.in_place and f.is_cuda and f.device == self.ctl.device and f.dtype in _X_DTYPES
                    and f.is_contiguous() and f.data_ptr() % 16 == 0 and r.is_cuda and r.is_contiguous()
                    and r.device == f.device):
                src, rows_ptr = f, r.data_ptr()      # rows gathered inside K0 / K23
                self._live_rows = r
            else:
                batch = batch.materialize()
        if rows_ptr:
            pass
        elif (self.in_place and batch.is_cuda and batch.device == self.ctl.device
                and batch.dtype in _X_DTYPES and batch.is_contiguous()
                and batch.data_ptr() % 16 == 0):
            src = batch                      # trained on where it lies
        elif self.in_place and batch.dtype != torch.float32:
            # a half batch from the host: staged in its own dtype (2 bytes per element over PCIe)
            src = self._xh.get(batch.dtype)
            if src is None:
                src = self._xh[batch.dtype] = torch.empty(tuple(batch.shape), dtype=batch.dtype,
                                                          device=self.ctl.device)
            src.copy_(batch, non_blocking=True)
        else:
            self.x.copy_(batch, non_blocking=True)   # converts a half batch to fp32 exactly
            src = self.x
        if src.dtype != self.x_dtype:        # switch to the captured graph of this dtype (if any)
            self._captured[self.x_dtype] = (self.graph, self._exec, self.kernels_per_replay)
            self.graph, self._exec, self.kernels_per_replay = self._captured.pop(src.dtype, (None, None, 0))
            self.x_dtype = src.dtype
        self._live = src                     # the caller may drop its reference before the replay runs
        self.x_slot_np[0] = src.data_ptr()
        self.rows_slot_np[0] = rows_ptr
        self.seq += 1
        self.seq_np[0] = self.seq
        group = tr.optimizer.param_groups[0]
        # AdamW state: created / re-laid-out on first use and whenever the optimizer's state objects were
        # replaced (load_state_dict); otherwise the cached numpy views of the `step` tensors are current
        opt_state = tr.optimizer.state
        if len(self._step_views) != len(self.params) or any(
                opt_state[p].get("step") is not tv[0] for p, tv in zip(self.params, self._step_views)):
            self._step_views = []
            for p in self.params:
                t = _ensure_adamw_state(tr.optimizer, p)["step"]
                self._step_views.append((t, None if t.is_cuda else t.numpy()))
            self.graph = None             # new state tensors: the captured moment pointers are void
            self._exec = None
            self._captured.clear()
        t0, v0 = self._step_views[0]
        step_t = float(v0 if v0 is not None else t0) + 1.0
        beta1, beta2 = group["betas"]
        h = self.hyper_np
        h[0], h[1], h[2], h[3], h[4] = group["lr"], beta1, beta2, group["eps"], group["weight_decay"]
        h[5] = 1.0 - beta1 ** step_t
        h[6] = math.sqrt(1.0 - beta2 ** step_t)
        h[7] = tr.config.gradient_clip
        ops.memcpy_async(self.ctl, self.ctl_host)      # 64 bytes, pinned -> device (raw cudaMemcpyAsync)
        self.calls += 1
        wd = tr.model.decoder.weight
        if wd.stride() != (1, wd.shape[0]):      # feature-major storage lost (.data assigned): re-point it
            tr.model._w_decT()
        key = self._pointer_key()
        if key != self._ptrs:      # storage was swapped behind our back (.data = ..., load): re-capture
            self.graph = None
            self._exec = None
            self._captured.clear()
            if self._ptrs:
                tr._dp_operands_fresh = False      # new weights: the gathered bf16 operands are void
            self._ptrs = key
            self.calls = 1
        if self.zero:
            self._operands()
            if not tr._dp_operands_fresh:
                if tr._dp_weights_stale:
                    raise RuntimeError("data parallel: the model's weights were replaced while this replica's "
                                       "fp32 rows were stale - call trainer.consolidate_weights() first")
                self._refresh_operands()
            tr._dp_weights_stale = True      # after this step the fp32 rows of other ranks are one step behind
        fresh = self.x_dtype not in self._warm     # this dtype's kernels have not run yet: one eager step
        self._warm.add(self.x_dtype)
        if self.calls > 1 and not fresh and tr.cuda_graph == "segments":
            # data parallel: the kernels between the collectives are four CUDA graphs (compute up to
            # dW_enc | dW_dec + b_pre gradient | counters + gradient norm | optimizer), the NCCL calls
            # stay eager between them (capturing them into one graph hung on the 2-GPU box in round 1)
            if self.graph is None:
                torch.cuda.synchronize()
                pool = torch.cuda.graph_pool_handle()
                before = ops.GPU_LAUNCHES
                segs = []
                for part in (self._compute_a, self._compute_b, self._update_pre, self._update_opt):
                    g = torch.cuda.CUDAGraph()
                    with _quiet_gc(), torch.cuda.graph(g, pool=pool):
                        part()
                    segs.append(g)
                self.kernels_per_replay = ops.GPU_LAUNCHES - before
                ops.GPU_LAUNCHES = before
                self.graph = segs
                self.captures += 1
            if not self._exec:        # raw cudaGraphExec_t handles of the four segments (see _launch_graph)
                self._exec = [self._raw_exec(g) for g in self.graph]
            launch = self._launch_one
            (ga, gb, gc, gd), (ea, eb, ec, ed) = self.graph, self._exec
            launch(ga, ea)
            if self._mid["use_gemm"]:
                self._start_early()
            launch(gb, eb)
            self._exchange()
            launch(gc, ec)
            if self.shard:
                tr.dp_comm.all_reduce_sum(self.sumsq)
            launch(gd, ed)
            if self.shard:
                self._gather_weights()
            ops.GPU_LAUNCHES += self.kernels_per_replay
        elif self.calls == 1 or fresh or tr.cuda_graph in ("eager", "segments"):
            self._body()
        else:
            if self.graph is None:
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                before = ops.GPU_LAUNCHES
                # data parallel (WSAE_DP_GRAPH=1): the NCCL watchdog thread queries events while this thread
                # captures - under the default "global" mode that alone invalidates the capture
                mode = "thread_local" if tr.data_parallel else "global"
                with _quiet_gc(), torch.cuda.graph(g, capture_error_mode=mode):
                    self._body()
                self.kernels_per_replay = ops.GPU_LAUNCHES - before   # captured, not yet executed
                ops.GPU_LAUNCHES = before
                self.graph = g
                self.captures += 1
                self._exec = None
            self._launch_graph()
            ops.GPU_LAUNCHES += self.kernels_per_replay
        # ---- host book-keeping, overlapping the kernels ----
        # torch.optim.AdamW keeps `step` as a CPU float32 tensor per parameter: bump them through
        # cached numpy views (re-made when a load_state_dict swapped the tensors)
        for t, view in self._step_views:
            if view is None:
                t += 1
            else:
                np.add(view, 1, out=view)
        tr.optimizer._opt_called = True    # the fused kernels ARE the optimizer step (lr_scheduler's order check)
        for p, g in zip(self.params, self._grad_views):   # expose grads the way autograd would
            if p.grad is not g:
                p.grad = g
        self.state.mailbox = self
        tr.model._last_sparse = self.state


class SAETrainer:
    """Trainer for sparse autoencoders (training.py:32-379)."""

    def __init__(
        self,
        model: TopKSAE,
        config: TrainingConfig,
        device: torch.device | str = "cpu",
        run_dir: Path | None = None,
        resample_dead_every: int = 5000,
        resample_batch_size: int = 8192,
        *,
        grad_scaler: bool = False,
        fused_optimizer: bool | None = None,
        cuda_graph: bool | None = None,
        auto_resample: bool = False,
        data_parallel: bool = False,
        dp_comm=None,
        global_batch_rows: int | None = None,
        project_decoder_grad: bool = False,
        deterministic: bool | None = None,
        shard_optimizer: bool | None = None,
    ):
        self.model = model.to(device)
        self.config = config
        self.device = device
        self.run_dir = run_dir or Path("outputs")
        self.run_dir.mkdir(parents=True, exist_ok=True)
        self.resample_dead_every = resample_dead_every
        self.resample_batch_size = resample_batch_size

        self.optimizer = AdamW(model.parameters(), lr=config.learning_rate,
                               weight_decay=config.weight_decay)
        self.scheduler = None

        is_cuda = str(device).startswith("cuda")
        self.use_amp = config.use_amp and is_cuda
        self.scaler = torch.amp.GradScaler("cuda", enabled=self.use_amp and grad_scaler)
        self.fused_optimizer = is_cuda if fused_optimizer is None else (fused_optimizer and is_cuda)

        self.global_step = 0
        self.epoch = 0
        self.metrics_history: list[TrainingMetrics] = []
        self.num_resampled_total = 0
        self.wandb_run = None
        self._resample_dataset = None
        self._hyper: Tensor | None = None
        self._sumsq: Tensor | None = None
        if cuda_graph is None:
            cuda_graph = os.environ.get("WSAE_CUDA_GRAPH", "1") != "0"
        # "eager": same kernel sequence as the captured graph, launched one by one (per-kernel timing)
        self.cuda_graph = cuda_graph if (cuda_graph and self.fused_optimizer
                                         and not self.scaler.is_enabled()) else False
        self._graphs: dict[int, _GraphedStep] = {}
        # batch-sharded data parallel (sae/parallel.py): every rank passes its own row shard to
        # train_step; gradients, stats and fired stamps are all-reduced inside the step
        # the reference defines _maybe_resample_dead_features but never calls it (training.py:97-134);
        # auto_resample=True wires it in after every step (off by default: parity)
        self.auto_resample = bool(auto_resample)
        # north_star's "gradient projection": remove the component of each decoder row's gradient along
        # the row before the AdamW step (fused into adamw_multi).  The reference does not do this
        # (grep finds no projection in sae/training.py), so it is OFF by default and excluded from parity.
        self.project_decoder_grad = bool(project_decoder_grad)
        # deterministic=True (or WSAE_DETERMINISTIC=1): the bf16 graphed step accumulates its cross-row
        # and split-K sums in a fixed / order-independent way (wsae_*_det), so two runs from the same
        # state are bit-identical; the default adds them with float atomics in arrival order
        if deterministic is None:
            deterministic = os.environ.get("WSAE_DETERMINISTIC", "0") == "1"
        self.deterministic = bool(deterministic)
        self.data_parallel = bool(data_parallel)
        # data parallel: reduce-scatter / sharded AdamW / all-gather instead of all-reduce + replicated
        # AdamW (sae/parallel.py); WSAE_DP_SHARD=0 or shard_optimizer=False keeps the replicated form
        if shard_optimizer is None:
            shard_optimizer = os.environ.get("WSAE_DP_SHARD", "1") != "0"
        self.shard_optimizer = bool(shard_optimizer)
        self.dp_comm = None
        self._dp_operands: tuple[Tensor, Tensor] | None = None   # bf16 operand gather (see _GraphedStep.zero)
        self._dp_operands_fresh = False
        self._dp_weights_stale = False
        self.global_batch_rows = global_batch_rows     # default: local rows x world (equal shards)
        if self.data_parallel:
            from .parallel import TorchDistCommunicator
            self.dp_comm = dp_comm if dp_comm is not None else TorchDistCommunicator()
            if not (is_cuda and self.fused_optimizer) or self.scaler.is_enabled():
                raise RuntimeError("data_parallel=True needs the fused CUDA step (no GradScaler)")
            # collectives between the kernels: four graph segments with eager NCCL calls between them (default).
            # WSAE_DP_GRAPH=1 captures the NCCL calls into ONE graph per step (measured on 2 GPUs: small
            # 2.38 -> 2.31 ms weak, 1.37 -> 1.33 ms strong; opt-in: the communicator must not be destroyed
            # while such a graph is alive - see _guard_process_group_teardown).
            graph_ok = getattr(self.dp_comm, "graph_safe", False) and \
                os.environ.get("WSAE_DP_GRAPH", "0") == "1" and self.cuda_graph is not False
            # default for real process groups: graph the kernel segments, keep the collectives eager
            seg_ok = getattr(self.dp_comm, "graph_safe", False) and self.cuda_graph is not False and \
                os.environ.get("WSAE_DP_SEGMENTS", "1") != "0"
            self.cuda_graph = True if graph_ok else ("segments" if seg_ok else "eager")
            if graph_ok:
                _guard_process_group_teardown(self)

    # ------------------------------------------------------------------ resampling plumbing
    def set_resample_dataset(self, dataset: torch.utils.data.Dataset) -> None:
        self._resample_dataset = dataset

    def _maybe_resample_dead_features(self) -> int:
        """Same gating as training.py:97-134 (the reference never calls it automatically either)."""
        if self._resample_dataset is None or not hasattr(self.model, "resample_dead_features"):
            return 0
        if self.global_step == 0 or self.global_step % self.resample_dead_every != 0:
            return 0
        self.consolidate_weights()
        picks = torch.randperm(len(self._resample_dataset))[: self.resample_batch_size]
        tensors = getattr(self._resample_dataset, "tensors", None)
        if tensors is not None:  # TensorDataset: one indexed gather instead of a Python loop
            batch = tensors[0][picks]
        else:
            rows = [self._resample_dataset[int(i)] for i in picks]
            rows = [r[0] if isinstance(r, tuple) else r for r in rows]
            batch = torch.stack(rows)
        batch = batch.to(self.device)
        if self.data_parallel:
            # replicas stay bit-identical only if every rank rewrites the same rows: rank 0's pick (its
            # RNG, its dataset shard) is broadcast; the resample forward itself is deterministic
            want = torch.tensor([batch.shape[0]], dtype=torch.int64, device=batch.device)
            self.dp_comm.broadcast(want)
            if batch.shape[0] != int(want):
                batch = torch.empty((int(want), batch.shape[1]), dtype=batch.dtype, device=batch.device)
            batch = self.dp_comm.broadcast(batch.contiguous())
        n = self.model.resample_dead_features(batch)
        self.num_resampled_total += n
        if n > 0 and self.wandb_run is not None:
            self.wandb_run.log({"train/features_resampled": n}, step=self.global_step)
        return n

    # ------------------------------------------------------------------ schedule
    def setup_scheduler(self, total_steps: int) -> None:
        """Linear warm-up (0.01 -> 1) then cosine to 0.1 * lr (training.py:136-159)."""
        warmup = min(self.config.warmup_steps, total_steps // 10)
        ramp = LinearLR(self.optimizer, start_factor=0.01, end_factor=1.0, total_iters=warmup)
        decay = CosineAnnealingLR(self.optimizer, T_max=total_steps - warmup,
                                  eta_min=self.config.learning_rate * 0.1)
        self.scheduler = SequentialLR(self.optimizer, schedulers=[ramp, decay], milestones=[warmup])

    # ------------------------------------------------------------------ optimizer step
    def _fused_clip_adamw(self) -> None:
        """clip_grad_norm_ + AdamW.step in len(params)+len(params) kernel launches, no host sync."""
        group = self.optimizer.param_groups[0]
        params = [p for p in group["params"] if p.grad is not None]
        if not params:
            return
        dev = params[0].device
        if self._sumsq is None:
            self._sumsq = torch.zeros(1, dtype=torch.float64, device=dev)
            self._hyper = torch.empty(8, dtype=torch.float32, device=dev)
        self._sumsq.zero_()
        for p in params:
            g = p.grad
            if not (g.is_contiguous() or g.t().is_contiguous()):
                p.grad = g = g.contiguous()
            ops.sumsq_(g, self._sumsq)
        # optimizer state, created exactly like torch.optim.AdamW does (step as a float32 tensor)
        step_t = None
        for p in params:
            state = _ensure_adamw_state(self.optimizer, p)
            state["step"] += 1
            step_t = float(state["step"])
        beta1, beta2 = group["betas"]
        lr = group["lr"]
        bc1 = 1.0 - beta1 ** step_t
        bc2s = math.sqrt(1.0 - beta2 ** step_t)
        hyper = torch.tensor([lr, beta1, beta2, group["eps"], group["weight_decay"], bc1, bc2s,
                              self.config.gradient_clip], dtype=torch.float32)
        self._hyper.copy_(hyper, non_blocking=True)
        self.optimizer._opt_called = True
        for p in params:
            state = self.optimizer.state[p]
            # parameter, grad and moments share one dense layout (contiguous or its transpose),
            # so a flat elementwise pass over the raw storage is exact
            if p.grad.stride() != p.stride():
                same_layout = torch.empty_strided(p.shape, p.stride(), dtype=p.dtype, device=p.device)
                p.grad = same_layout.copy_(p.grad)
            ops.fused_adamw_(p.data, p.grad, state["exp_avg"], state["exp_avg_sq"], self._hyper,
                             self._sumsq)

    # ------------------------------------------------------------------ the hot loop
    def train_step(self, batch: Tensor | tuple | list) -> TrainingMetrics:
        """One optimisation step; same order of operations as training.py:161-217."""
        if not self.model.training:      # model.train() walks every submodule: 10+ us of the ~60 us YAML-batch step
            self.model.train()
        if isinstance(batch, (tuple, list)):
            batch = batch[0]
        graph_ok = self._graph_ok(batch)
        if isinstance(batch, IndexedBatch) and not graph_ok:
            batch = batch.materialize()      # only the graphed step gathers rows inside its kernels
        if self.data_parallel:
            if not graph_ok:
                raise RuntimeError("data_parallel=True supports the fused TopKSAE step only")
            self.model._global_rows = self.global_batch_rows or batch.shape[0] * self.dp_comm.world
        if graph_ok:
            gs = self._graphs.get(batch.shape[0])
            if gs is None:
                gs = self._graphs[batch.shape[0]] = _GraphedStep(self, batch.shape[0])
            gs.run(batch)
            if self.scheduler is not None:
                self.scheduler.step()
            self.global_step += 1
            metrics = self._read_metrics(None, batch.shape[0])
            if self.auto_resample:
                self._maybe_resample_dead_features()
            return metrics

        batch = batch.to(self.device, non_blocking=True)

        # bf16, not torch's fp16 default: the scaler is disabled unless grad_scaler=True, and models that
        # do not run through the fused node (ReLUSAE, dense crosscoders, SkipTranscoder.skip) would train
        # in fp16 without loss scaling otherwise; with an ENABLED scaler the reference's fp16 is kept
        amp_dtype = torch.float16 if self.scaler.is_enabled() else torch.bfloat16
        with torch.amp.autocast("cuda", enabled=self.use_amp, dtype=amp_dtype):
            output: SAEOutput = self.model(batch)

        self.optimizer.zero_grad()
        self.scaler.scale(output.loss).backward()

        if self.fused_optimizer and not self.scaler.is_enabled():
            self._fused_clip_adamw()
        else:
            self.scaler.unscale_(self.optimizer)
            torch.nn.utils.clip_grad_norm_(self.model.parameters(), self.config.gradient_clip)
            self.scaler.step(self.optimizer)
            self.scaler.update()

        if hasattr(self.model, "normalize_decoder_weights"):
            self.model.normalize_decoder_weights()
        if self.scheduler is not None:
            self.scheduler.step()
        self.global_step += 1

        metrics = self._read_metrics(output, batch.shape[0])
        if self.auto_resample:
            self._maybe_resample_dead_features()
        return metrics

    def _graph_ok(self, batch: Tensor) -> bool:
        m = self.model
        if not (self.cuda_graph and isinstance(m, TopKSAE) and type(m).forward is TopKSAE.forward
                and batch.dim() == 2 and batch.shape[1] == m.input_dim and m.input_dim % 4 == 0
                and batch.dtype in _X_DTYPES and m.k <= GRAPH_MAX_K
                and ops.bucket_supported(m.hidden_dim, m.k) and m.precision is None):
            return False
        # the five parameters by attribute (Module.parameters() walks the module tree: ~10 us per call)
        return (m.b_pre.requires_grad and m.encoder.weight.requires_grad and m.encoder.bias.requires_grad
                and m.decoder.weight.requires_grad and m.decoder.bias.requires_grad)

    def _read_metrics(self, output: SAEOutput | None, rows: int) -> TrainingMetrics:
        lr = self.optimizer.param_groups[0]["lr"]
        st = getattr(self.model, "_last_sparse", None)
        if st is not None and st.stats is not None and (output is None or output.loss.is_cuda):
            if output is None and getattr(st, "mailbox", None) is not None:
                # graphed step: the counters kernel posted the 24 bytes to pinned memory - no stream sync
                sse, l0_count, dead_count = st.mailbox.wait_metrics()
            else:
                raw = st.stats.cpu()  # the step's single device->host sync (24 bytes)
                sse = raw[:1].view(torch.float64).item()
                l0_count, dead_count = raw[1].item(), raw[2].item()
            # the reference's metrics are fp32 tensors read with .item(): round the same way
            d_out = st.d_out
            loss = float(np.float32(sse / (float(st.rows_total) * d_out)))
            l0_rows = st.rows_total if self.data_parallel else rows
            l0 = float(np.float32(l0_count / float(l0_rows)))
            hidden_dim = self.model.feature_last_activated.numel()
            dead = float(np.float32(dead_count) / np.float32(hidden_dim))
            return TrainingMetrics(loss, loss, 0.0, l0, dead, lr, self.global_step)
        return TrainingMetrics(
            loss=output.loss.item(),
            reconstruction_loss=output.reconstruction_loss.item(),
            sparsity_loss=output.sparsity_loss.item(),
            l0=output.l0.item(),
            dead_feature_ratio=self.model.get_dead_feature_ratio(),
            learning_rate=lr,
            step=self.global_step,
        )

    def _prefetched(self, dataloader):
        """Iterate ``dataloader`` one batch ahead: the host->device copy of batch n+1 is issued on a
        side stream before step n runs, so PCIe traffic hides behind compute (pinned batches, which
        is what ``FeatureCache.get_dataloader`` yields with ``pin_memory=True``)."""
        if not str(self.device).startswith("cuda"):
            yield from dataloader
            return
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)

        def stage(item):
            t = item[0] if isinstance(item, (tuple, list)) else item
            if t.is_cuda:
                return t, None
            with torch.cuda.stream(self._copy_stream):
                dev = t.to(self.device, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self._copy_stream)
            return dev, ev

        it = iter(dataloader)
        try:
            ahead = stage(next(it))
        except StopIteration:
            return
        while ahead is not None:
            dev, ev = ahead
            try:
                ahead = stage(next(it))
            except StopIteration:
                ahead = None
            if ev is not None:
                main = torch.cuda.current_stream()
                main.wait_event(ev)
                dev.record_stream(main)
            yield dev

    def train_epoch(self, dataloader: DataLoader, progress: Progress | None = None,
                    task_id: int | None = None) -> list[TrainingMetrics]:
        epoch_metrics: list[TrainingMetrics] = []
        for batch in self._prefetched(dataloader):
            m = self.train_step(batch)
            epoch_metrics.append(m)
            self.metrics_history.append(m)
            if progress is not None and task_id is not None:
                progress.update(task_id, advance=1)
            if self.wandb_run is not None and self.global_step % 100 == 0:
                self.wandb_run.log(
                    {"train/loss": m.loss, "train/reconstruction_loss": m.reconstruction_loss,
                     "train/l0": m.l0, "train/dead_ratio": m.dead_feature_ratio,
                     "train/lr": m.learning_rate},
                    step=self.global_step,
                )
        self.consolidate_weights()
        self.epoch += 1
        return epoch_metrics

    def train(self, dataloader: DataLoader, epochs: int | None = None,
              checkpoint_every: int | None = None) -> None:
        epochs = epochs or self.config.epochs
        checkpoint_every = checkpoint_every or self.config.checkpoint_every
        self.setup_scheduler(len(dataloader) * epochs)
        columns = (SpinnerColumn(), TextColumn("[progress.description]{task.description}"),
                   BarColumn(), TaskProgressColumn())
        with Progress(*columns) as progress:
            outer = progress.add_task(f"[cyan]Training {epochs} epochs", total=epochs)
            for e in range(epochs):
                inner = progress.add_task(f"[green]Epoch {e + 1}/{epochs}", total=len(dataloader))
                ms = self.train_epoch(dataloader, progress, inner)
                mean_loss = sum(m.loss for m in ms) / len(ms)
                mean_l0 = sum(m.l0 for m in ms) / len(ms)
                progress.remove_task(inner)
                progress.update(outer, advance=1)
                progress.console.print(
                    f"Epoch {e + 1}: loss={mean_loss:.4f}, L0={mean_l0:.1f}, "
                    f"dead={ms[-1].dead_feature_ratio:.1%}"
                )
                if (e + 1) % checkpoint_every == 0:
                    self.save_checkpoint(f"checkpoint_epoch{e + 1}.pt")
        self.save_checkpoint("final.pt")

    # ------------------------------------------------------------------ persistence
    def save_checkpoint(self, filename: str) -> Path:
        """Same dict layout as training.py:328-338."""
        path = self.run_dir / filename
        self.consolidate_weights()
        self.consolidate_optimizer_state()
        payload = {
            "model_state_dict": self.model.state_dict(),
            "optimizer_state_dict": self.optimizer.state_dict(),
            "scheduler_state_dict": self.scheduler.state_dict() if self.scheduler else None,
            "global_step": self.global_step,
            "epoch": self.epoch,
            "config": self.config.model_dump(),
        }
        torch.save(payload, path)
        return path

    def release_graphs(self) -> None:
        """Drop the captured CUDA graphs (they are re-captured on the next step).  Call it before
        ``torch.distributed.destroy_process_group()`` when the step's NCCL collectives are captured into
        the graph (``WSAE_DP_GRAPH=1``): destroying the communicator while graphs that hold its kernels
        are alive blocks forever."""
        for gs in self._graphs.values():
            gs.graph = None
            gs._exec = None
            gs._captured.clear()
        self._graphs.clear()
        gc.collect()
        if str(self.device).startswith("cuda"):
            torch.cuda.synchronize(self.device)

    def consolidate_weights(self) -> None:
        """Data parallel with the bf16 operand gather: a replica keeps only ITS feature rows of the fp32
        encoder / decoder weights current between steps (the step itself reads the gathered bf16
        operands).  This gathers the fp32 rows into every replica - call it before reading or editing
        ``model``'s weights (collective: every rank calls it; ``train_epoch``, ``save_checkpoint`` and
        the resampling hook do).  A no-op otherwise."""
        if self.dp_comm is None or not self._dp_weights_stale:
            return
        m = self.model
        self.dp_comm.all_gather_rows(m.encoder.weight.data)
        self.dp_comm.all_gather_rows(m.decoder.weight.data.t())
        self._dp_weights_stale = False
        self._dp_operands_fresh = False      # the caller may edit the weights now: re-pack before the next step

    def consolidate_optimizer_state(self) -> None:
        """Sharded optimizer: every rank updates the AdamW moments of ITS feature rows only; gather the
        rows so that ``optimizer.state_dict()`` is complete on every rank (collective: all ranks call it).
        A no-op otherwise."""
        gs = next((g for g in self._graphs.values() if getattr(g, "shard", False)), None)
        if gs is None:
            return
        m = self.model
        for p in (m.encoder.weight, m.decoder.weight):
            st = self.optimizer.state.get(p)
            if not st:
                continue
            for name in ("exp_avg", "exp_avg_sq"):
                t = st[name].t() if p is m.decoder.weight else st[name]
                self.dp_comm.all_gather_rows(t)

    def load_checkpoint(self, path: str | Path) -> None:
        ckpt = torch.load(path, map_location=self.device)
        self.model.load_state_dict(ckpt["model_state_dict"])
        self._dp_weights_stale = False
        self._dp_operands_fresh = False
        self.optimizer.load_state_dict(ckpt["optimizer_state_dict"])
        if ckpt["scheduler_state_dict"] and self.scheduler:
            self.scheduler.load_state_dict(ckpt["scheduler_state_dict"])
        self.global_step = ckpt["global_step"]
        self.epoch = ckpt["epoch"]

    def save_metrics(self, filename: str = "metrics.json") -> Path:
        path = self.run_dir / filename
        keys = ("step", "loss", "reconstruction_loss", "sparsity_loss", "l0",
                "dead_feature_ratio", "learning_rate")
        rows = [{k: asdict(m)[k] for k in keys} for m in self.metrics_history]
        path.write_text(json.dumps(rows, indent=2))
        return path
