"""Tensor-level wrappers over the C ABI (``include/wsae.h``).

PyTorch is used only for device memory and streams: every function here checks dtypes/layouts,
passes raw device pointers + the current CUDA stream into ``libwsae_sm100.so`` and returns torch
tensors.  CPU tensors are rejected — there is deliberately no CPU fallback.
"""

from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass

import torch
from torch import Tensor

from . import _lib

GPU_LAUNCHES = 0  # kernels launched through this module (bench.py reports it)


_RAW_STREAM = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream() -> int:
    """cudaStream_t of torch's current stream on the current device (the raw C getter: the Python
    `torch.cuda.current_stream()` wrapper costs ~8 us per call, which the 60 us YAML-batch step notices)."""
    if _RAW_STREAM is not None:
        return _RAW_STREAM(torch._C._cuda_getDevice())
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def _need_cuda(*tensors: Tensor | None) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "whisper_sae_b200 kernels run on CUDA (sm_100a) tensors only; there is no CPU "
                "fallback (got a tensor on %s)" % t.device
            )


def _f32c(t: Tensor | None, name: str) -> None:
    if t is None:
        return
    if t.dtype != torch.float32 or not t.is_contiguous():
        raise RuntimeError(f"{name} must be a contiguous float32 tensor")


# activation element types the kernels read, by the C ABI's dtype code (include/wsae.h)
_LN_DTYPES = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}


def _x_dtype_code(dtype: torch.dtype) -> int:
    if dtype not in _LN_DTYPES:
        raise RuntimeError(f"unsupported activation dtype {dtype} (float32, bfloat16 or float16)")
    return _LN_DTYPES[dtype]


def _check_slot(slot: Tensor, name: str) -> None:
    if slot.dtype != torch.int64 or slot.numel() != 1 or not slot.is_cuda:
        raise RuntimeError(f"{name} must be a one-element int64 CUDA tensor holding a device address")


def _count(n: int = 1) -> None:
    global GPU_LAUNCHES
    GPU_LAUNCHES += n


class KernelProfile:
    """Per-kernel CUDA-event timing on the launching stream (enabled by bench.py for one pass)."""

    def __init__(self) -> None:
        self.spans: dict[str, list[tuple[torch.cuda.Event, torch.cuda.Event]]] = {}

    def summary(self) -> dict[str, dict[str, float]]:
        torch.cuda.synchronize()
        out = {}
        for name, spans in self.spans.items():
            ms = [a.elapsed_time(b) for a, b in spans]
            out[name] = {"launches": len(ms), "total_ms": sum(ms), "avg_ms": sum(ms) / max(1, len(ms))}
        return out


PROFILE: KernelProfile | None = None


def _run(name: str, fn, *args, launches: int = 1) -> None:
    """Call one C-ABI entry point, raise on a non-zero status, count (and optionally time) it."""
    prof = PROFILE
    if prof is None:
        _lib.check(fn(*args), name)
    else:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        _lib.check(fn(*args), name)
        b.record()
        prof.spans.setdefault(name, []).append((a, b))
    _count(launches)


@dataclass(frozen=True)
class PackedShape:
    d: int
    terms: int
    dp: int
    used_cols: int
    kp: int


def packed_shape(d: int, terms: int) -> PackedShape:
    lib = _lib.load()
    dp, used, kp = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    _lib.check(lib.wsae_packed_k(d, terms, ctypes.byref(dp), ctypes.byref(used), ctypes.byref(kp)),
               "wsae_packed_k")
    return PackedShape(d, terms, dp.value, used.value, kp.value)


def _round_up(a: int, b: int) -> int:
    return (a + b - 1) // b * b


def pack_activations(x: Tensor, b_pre: Tensor | None, terms: int, out: Tensor | None = None) -> Tensor:
    _need_cuda(x, b_pre)
    _f32c(x, "x")
    _f32c(b_pre, "b_pre")
    B, d = x.shape
    ps = packed_shape(d, terms)
    Bp = _round_up(B, 128)
    if out is None or out.shape != (Bp, ps.kp):
        out = torch.empty((Bp, ps.kp), dtype=torch.bfloat16, device=x.device)
    lib = _lib.load()
    _run("wsae_pack_activations", lib.wsae_pack_activations, _ptr(x), _ptr(b_pre), B, Bp, d, terms, _ptr(out), _stream())
    return out


def pack_activations_at(x_at: Tensor, B: int, d: int, b_pre: Tensor | None,
                        out: Tensor | None = None, rows_at: Tensor | None = None,
                        x_dtype: torch.dtype = torch.float32) -> Tensor:
    """``pack_activations`` (bf16, one term) of the ``[B, d]`` matrix whose device address the int64
    slot ``x_at`` holds WHEN THE KERNEL RUNS (graph replay on batches in place).  ``x_dtype``: its
    element type (float32, bfloat16 or float16; a slot holds only an address).  ``rows_at``: a second
    int64 slot holding the address of an int64 row-index array (0 = identity): batch row r is row
    ``rows[r]`` of the matrix (shuffled batches of a resident matrix, never materialised)."""
    _need_cuda(x_at, b_pre, rows_at)
    _f32c(b_pre, "b_pre")
    _check_slot(x_at, "x_at")
    if rows_at is not None:
        _check_slot(rows_at, "rows_at")
    ps = packed_shape(d, 1)
    Bp = _round_up(B, 128)
    if out is None or out.shape != (Bp, ps.kp):
        out = torch.empty((Bp, ps.kp), dtype=torch.bfloat16, device=x_at.device)
    lib = _lib.load()
    _run("wsae_pack_activations", lib.wsae_pack_activations_typed, _ptr(x_at), _ptr(rows_at), _x_dtype_code(x_dtype),
         _ptr(b_pre), B, Bp, d, 1, _ptr(out), _stream())
    return out


def pack_encoder(w_enc: Tensor, b_enc: Tensor | None, terms: int, out: Tensor | None = None) -> Tensor:
    _need_cuda(w_enc, b_enc)
    _f32c(w_enc, "encoder.weight")
    _f32c(b_enc, "encoder.bias")
    F, d = w_enc.shape
    ps = packed_shape(d, terms)
    Fp = _round_up(F, 256)
    if out is None or out.shape != (Fp, ps.kp):
        out = torch.empty((Fp, ps.kp), dtype=torch.bfloat16, device=w_enc.device)
    lib = _lib.load()
    _run("wsae_pack_encoder", lib.wsae_pack_encoder, _ptr(w_enc), _ptr(b_enc), F, Fp, d, terms, _ptr(out), _stream())
    return out


def pack_encoder_rows_(w_rows: Tensor, b_rows: Tensor | None, terms: int, out_rows: Tensor) -> None:
    """K0 on a block of feature rows: packs ``w_rows`` [R, d] (+ bias) into the matching rows of a packed
    encoder matrix (``out_rows`` = a row slice of it, [R, Kp] bf16) without touching any padding rows -
    what a rank of the sharded optimizer does with the rows it has just updated."""
    _need_cuda(w_rows, b_rows, out_rows)
    _f32c(w_rows, "encoder.weight rows")
    _f32c(b_rows, "encoder.bias rows")
    R, d = w_rows.shape
    ps = packed_shape(d, terms)
    if out_rows.dtype != torch.bfloat16 or tuple(out_rows.shape) != (R, ps.kp) or not out_rows.is_contiguous():
        raise RuntimeError(f"out_rows must be a contiguous [{R}, {ps.kp}] bfloat16 row block")
    lib = _lib.load()
    _run("wsae_pack_encoder", lib.wsae_pack_encoder, _ptr(w_rows), _ptr(b_rows), R, R, d, terms, _ptr(out_rows), _stream())


_SM_COUNT: dict[int, int] = {}


def sm_count(device: torch.device) -> int:
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _SM_COUNT:
        _SM_COUNT[idx] = torch.cuda.get_device_properties(idx).multi_processor_count
    return _SM_COUNT[idx]


def choose_nsplit(B: int, F: int, k: int, num_sms: int) -> int:
    """Pick the F-split count that minimises (waves x tiles per split) for the persistent grid."""
    m_blocks = (B + 127) // 128
    n_tiles = (F + 255) // 256
    best, best_cost = 1, None
    for ns in range(1, n_tiles + 1):
        tps = (n_tiles + ns - 1) // ns
        ns_eff = (n_tiles + tps - 1) // tps
        if ns_eff != ns:
            continue
        if ns > 1 and (ns * k + 31) // 32 > 64:
            break
        waves = (m_blocks * ns + num_sms - 1) // num_sms
        # every work item pays a fixed start-up cost (the running threshold restarts at -inf and the
        # first few hundred columns are almost all accepted): measured ~8 tile-times per item
        cost = waves * (tps + 8) + (0.15 * ns if ns > 1 else 0.0)
        if best_cost is None or cost < best_cost - 1e-9:
            best, best_cost = ns, cost
    return best


# rows up to which K1 runs as dense GEMM + row-wise select (wsae_encode_topk_dense); 0 switches it off
_DENSE_ROWS = int(os.environ.get("WSAE_K1_DENSE_ROWS", "1024"))
# the fused TopK epilogues of wsae_encode_topk keep at most 64 candidates per row
ENCODE_FUSED_MAX_K = 64
# scratch per chunk of the chunked route (fp32 pre-activations, plus the sliced select's candidate lists
# above 49 152 features): written by the GEMM and read back by the select while it is still in L2 (126 MB
# on a B200)
_CHUNK_SCRATCH_BYTES = 40 << 20
# the row select holds one row's keys in shared memory: wider rows are selected in column slices of at
# most this many features, whose k candidates each a merge reduces to k (wsae_encode_topk_chunked)
_SELECT_MAX_COLS = 49152


def encode_route(B: int, F: int, k: int, nsplit: int | None = None) -> str:
    """The K1 form ``encode_topk`` runs: "dense" (one GEMM storing [B, F] + one block per row
    selecting, batches <= WSAE_K1_DENSE_ROWS, F <= 49152, F % 4 == 0), "chunked" (the same over row
    chunks, at any F: every k > 64 that "dense" does not take) or "fused" (the GEMM with the TopK in its
    epilogue, k <= 64)."""
    dense_ok = F <= _SELECT_MAX_COLS and F % 4 == 0
    if nsplit is None and B <= _DENSE_ROWS and dense_ok:
        return "dense"
    if k > ENCODE_FUSED_MAX_K:
        return "chunked"
    return "fused"


def encode_chunk_scratch_floats(F: int, k: int, rows: int) -> int:
    """fp32 words of scratch the chunked route needs for ``rows`` rows per chunk: the pre-activations
    at row pitch round_up(F, 4), and above 49 152 features the [rows, nslices * k] candidate values and
    indices of the sliced select."""
    nslices = (F + _SELECT_MAX_COLS - 1) // _SELECT_MAX_COLS
    return rows * (_round_up(F, 4) + (2 * nslices * k if nslices > 1 else 0))


def encode_chunk_rows(B: int, F: int, k: int = 256) -> int:
    """Rows per chunk of the chunked K1 route: a multiple of 128 whose scratch fits
    _CHUNK_SCRATCH_BYTES, no more than the batch needs.  ``k`` sizes the candidate lists of the sliced
    select above 49 152 features (by default for k = 256, the largest k of the graphed step); at most
    49 152 features the scratch does not depend on it."""
    rows = max(128, _CHUNK_SCRATCH_BYTES // (4 * encode_chunk_scratch_floats(F, k, 1)) // 128 * 128)
    return min(rows, _round_up(B, 128))


def encode_topk(a_packed: Tensor, w_packed: Tensor, B: int, F: int, d: int, terms: int, k: int,
                nsplit: int | None = None) -> tuple[Tensor, Tensor]:
    """K1. Returns (idx int32 [B,k], val float32 [B,k]) — signed pre-activations, unordered."""
    _need_cuda(a_packed, w_packed)
    if k > F:
        raise RuntimeError(f"selected index k out of range (k={k} > hidden_dim={F})")
    ps = packed_shape(d, terms)
    Bp, Fp = a_packed.shape[0], w_packed.shape[0]
    lib = _lib.load()
    dev = a_packed.device
    route = encode_route(B, F, k, nsplit)
    idx = torch.empty((B, k), dtype=torch.int32, device=dev)
    val = torch.empty((B, k), dtype=torch.float32, device=dev)
    if route == "dense":
        # small batches (the shipped YAML batch is 128 rows): dense pre-activations + one block per row
        pre = torch.empty((B, F), dtype=torch.float32, device=dev)
        _run("wsae_encode_topk", lib.wsae_encode_topk_dense, _ptr(a_packed), _ptr(w_packed), B, Bp, F, Fp, ps.kp, ps.used_cols, k, _ptr(pre), _ptr(val), _ptr(idx), _stream(), launches=2)
        return idx, val
    if route == "chunked":
        # the scratch is allocated per call: inside a captured train step it belongs to the graph
        rows = encode_chunk_rows(B, F, k)
        pre = torch.empty(encode_chunk_scratch_floats(F, k, rows), dtype=torch.float32, device=dev)
        _run("wsae_encode_topk_chunked", lib.wsae_encode_topk_chunked, _ptr(a_packed), _ptr(w_packed), B, Bp, F, Fp, ps.kp, ps.used_cols, k, rows, _ptr(pre), _ptr(val), _ptr(idx), _stream(), launches=2 * ((B + rows - 1) // rows))
        return idx, val
    if nsplit is None:
        nsplit = choose_nsplit(B, F, k, sm_count(dev))
    nsplit = lib.wsae_encode_effective_splits(F, nsplit)
    pv = pi = None
    if nsplit > 1:
        pv = torch.empty((B, nsplit * k), dtype=torch.float32, device=dev)
        pi = torch.empty((B, nsplit * k), dtype=torch.int32, device=dev)
    _run("wsae_encode_topk", lib.wsae_encode_topk, _ptr(a_packed), _ptr(w_packed), B, Bp, F, Fp, ps.kp, ps.used_cols, k, nsplit, _ptr(pv), _ptr(pi), _ptr(val), _ptr(idx), _stream(), launches=2 if nsplit > 1 else 1)
    return idx, val


def decode_mse(target: Tensor, w_decT: Tensor, b_dec: Tensor, b_pre: Tensor | None, idx: Tensor,
               val: Tensor, *, want_resid: bool = True, want_recon: bool = False,
               stats: Tensor | None = None, last_activated: Tensor | None = None,
               step_count: Tensor | None = None) -> tuple[Tensor | None, Tensor | None]:
    """K2. ``stats`` is an int64[>=2] tensor: [0] holds a float64 SSE (bit pattern), [1] the L0 count."""
    _need_cuda(target, w_decT, b_dec, b_pre, idx, val, stats, last_activated, step_count)
    _f32c(target, "target")
    _f32c(b_dec, "decoder.bias")
    _f32c(b_pre, "b_pre")
    F, d = w_decT.shape
    B, k = idx.shape
    if not w_decT.is_contiguous() or w_decT.dtype not in (torch.float32, torch.bfloat16):
        raise RuntimeError("w_decT must be contiguous [F, d] float32 or bfloat16")
    resid = torch.empty_like(target) if want_resid else None
    recon = torch.empty_like(target) if want_recon else None
    lib = _lib.load()
    _run("wsae_decode_mse", lib.wsae_decode_mse, _ptr(target), _ptr(w_decT), int(w_decT.dtype == torch.bfloat16), _ptr(b_dec), _ptr(b_pre), _ptr(idx), _ptr(val), B, d, F, k, _ptr(resid), _ptr(recon), _ptr(stats), _ptr(last_activated), _ptr(step_count), _stream())
    return resid, recon


def backward_sparse(resid: Tensor, x: Tensor | None, b_pre: Tensor | None, w_decT: Tensor,
                    idx: Tensor, val: Tensor, grad_out: Tensor | None, coef: float, *,
                    d_w_enc: Tensor | None, d_w_decT: Tensor | None, d_b_enc: Tensor | None,
                    d_b_dec: Tensor | None, dpre_val: Tensor | None,
                    resid_bf16: Tensor | None = None) -> None:
    """K3. Accumulates into the provided (pre-zeroed) gradient buffers; ``d_w_enc``/``d_w_decT`` =
    None skips the weight-gradient scatters (the tensor-core K4 path computes them instead)."""
    _need_cuda(resid, x, w_decT, idx, val, grad_out)
    F, d = w_decT.shape
    B, k = idx.shape
    if d % 4 != 0:
        raise RuntimeError("input_dim must be a multiple of 4 for the sparse backward kernels")
    lib = _lib.load()
    _run("wsae_backward_sparse", lib.wsae_backward_sparse, _ptr(resid), _ptr(x), _ptr(b_pre), _ptr(w_decT), int(w_decT.dtype == torch.bfloat16), _ptr(idx), _ptr(val), _ptr(grad_out), float(coef), B, d, F, k, _ptr(d_w_enc), _ptr(d_w_decT), _ptr(d_b_enc), _ptr(d_b_dec), _ptr(dpre_val), _ptr(resid_bf16), _stream())


def memcpy_async(dst: Tensor, src: Tensor) -> None:
    """cudaMemcpyAsync of ``src`` (pinned host or device, contiguous) into ``dst`` on the current stream."""
    n = src.numel() * src.element_size()
    if n != dst.numel() * dst.element_size():
        raise RuntimeError("memcpy_async: size mismatch")
    lib = _lib.load()
    _lib.check(lib.wsae_memcpy_async(dst.data_ptr(), src.data_ptr(), n, _stream()), "wsae_memcpy_async")


def graph_launch(graph_exec: int) -> None:
    """cudaGraphLaunch(graph_exec, current stream) through the library (see SAETrainer's graphed step)."""
    lib = _lib.load()
    _lib.check(lib.wsae_graph_launch(graph_exec, _stream()), "wsae_graph_launch")


def row_step_supported(B: int, d: int, F: int, k: int, bf16: bool) -> bool:
    """Shapes the one-block-per-row small-batch step covers (else: K1 selection + K23 + bucket + K4)."""
    return (bf16 and B <= int(os.environ.get("WSAE_ROW_STEP_ROWS", "512")) and k <= 32 and d % 8 == 0
            and F % 4 == 0 and (F + 2 * d) * 4 <= 200 * 1024)


def encode_dense(a_packed: Tensor, w_packed: Tensor, B: int, F: int, d: int, terms: int,
                 out: Tensor | None = None) -> Tensor:
    """The GEMM of K1 alone: dense pre-activations [B, F] fp32 (small batches: L2-sized scratch)."""
    _need_cuda(a_packed, w_packed)
    ps = packed_shape(d, terms)
    if a_packed.dtype != torch.bfloat16 or a_packed.shape[1] != ps.kp or w_packed.shape[1] != ps.kp:
        raise RuntimeError("packed operands do not match (d, terms)")
    if out is None:
        out = torch.empty((B, F), dtype=torch.float32, device=a_packed.device)
    lib = _lib.load()
    _run("wsae_encode_topk", lib.wsae_encode_dense, _ptr(a_packed), _ptr(w_packed), B, a_packed.shape[0], F,
         w_packed.shape[0], ps.kp, ps.used_cols, _ptr(out), _stream())
    return out


def row_step(pre: Tensor, target: Tensor, w_decT: Tensor, b_dec: Tensor, b_pre: Tensor | None,
             grad_out: Tensor | None, coef: float, k: int, *, stats: Tensor | None,
             last_activated: Tensor | None, step_count: Tensor | None, d_b_enc: Tensor | None,
             d_b_dec: Tensor | None, d_w_enc: Tensor | None, d_w_decT: Tensor | None,
             resid: Tensor | None = None, dpre_val: Tensor | None = None, target_is_slot: bool = False,
             rows_at: Tensor | None = None, w_enc: Tensor | None = None,
             d_b_pre: Tensor | None = None,
             finish: tuple[Tensor, int, Tensor | None, Tensor, Tensor] | None = None,
             x_dtype: torch.dtype = torch.float32) -> tuple[Tensor, Tensor]:
    """Small-batch step, one block per row: TopK of ``pre`` + sparse decode + MSE + stamps + dv + bias
    gradients + both weight-gradient rows (fp32 atomics).  Returns (idx int32 [B,k], val fp32 [B,k]).
    The target is float32, bfloat16 or float16: its own dtype, or ``x_dtype`` when it is a slot."""
    _need_cuda(pre, target, w_decT, b_dec, b_pre, grad_out)
    _f32c(pre, "pre")
    B, F = pre.shape
    d = w_decT.shape[1]
    if w_decT.dtype != torch.bfloat16 or not w_decT.is_contiguous() or w_decT.shape[0] != F:
        raise RuntimeError("w_decT must be contiguous [F, d] bfloat16")
    if target_is_slot:
        _check_slot(target, "target slot")
        tgt, tgt_at = None, target
    else:
        if not target.is_contiguous():
            raise RuntimeError("target must be contiguous")
        tgt, tgt_at, x_dtype = target, None, target.dtype
    idx = torch.empty((B, k), dtype=torch.int32, device=pre.device)
    val = torch.empty((B, k), dtype=torch.float32, device=pre.device)
    lib = _lib.load()
    # finish = (ticket: zeroed 4+ bytes on the device, dead threshold, dead_count int64[1] | None, seq int64[1]
    # on the device, mailbox: 4 x int64 pinned host): the last block also bumps step_count and posts the metrics
    fin = (None, 0, None, None, None)
    if finish is not None:
        ticket, thr, dead, seq, mailbox = finish
        fin = (_ptr(ticket), int(thr), _ptr(dead), _ptr(seq), _ptr(mailbox))
    _run("wsae_row_step", lib.wsae_row_step_typed, _ptr(pre), _ptr(tgt), _ptr(tgt_at), _ptr(rows_at), _x_dtype_code(x_dtype), _ptr(w_decT),
         _ptr(b_dec), _ptr(b_pre), _ptr(grad_out), float(coef), B, d, F, k, _ptr(val), _ptr(idx), _ptr(stats),
         _ptr(last_activated), _ptr(step_count), _ptr(d_b_enc), _ptr(d_b_dec), _ptr(d_w_enc), _ptr(d_w_decT),
         _ptr(resid), _ptr(dpre_val), _ptr(w_enc), _ptr(d_b_pre), *fin, _stream())
    return idx, val


# largest k of the team-of-warps K23 (wsae_decode_backward.cu, wide form)
DECODE_BACKWARD_MAX_K = 256


def decode_backward_supported(d: int, k: int, bf16: bool, deterministic: bool = False) -> bool:
    """Shapes covered by the fused K23 kernels (else: decode_mse + backward_sparse): k <= 32 with
    d % 8 == 0, and 64 < k <= 256 with d % 128 == 0 (the team-of-warps form).  33 <= k <= 64 stays on
    K2 + K3 unless WSAE_WIDE_K23=1 routes it to the team form too.  ``deterministic``: the shapes of
    the deterministic form (``det_ws``), which has no K2 + K3 counterpart, so 33 <= k <= 64 takes the
    team form whatever WSAE_WIDE_K23 says."""
    if not (bf16 and d % 8 == 0 and os.environ.get("WSAE_FUSED_DECODE", "1") != "0"):
        return False
    if k <= 32:
        return True
    if d % 128 != 0 or k > DECODE_BACKWARD_MAX_K:
        return False
    return deterministic or k > 64 or os.environ.get("WSAE_WIDE_K23", "0") == "1"


def decode_backward(target: Tensor, w_decT: Tensor, b_dec: Tensor, b_pre: Tensor | None,
                    idx: Tensor, val: Tensor, grad_out: Tensor | None, coef: float, *,
                    resid: Tensor | None, resid_bf16: Tensor | None, stats: Tensor | None,
                    last_activated: Tensor | None, step_count: Tensor | None,
                    d_b_enc: Tensor | None, d_b_dec: Tensor | None, dpre_val: Tensor | None,
                    target_is_slot: bool = False, rows_at: Tensor | None = None,
                    det_ws: Tensor | None = None, x_dtype: torch.dtype = torch.float32) -> None:
    """K23: sparse decode + MSE + L0 + fired stamps + dv / bias gradients in one pass.
    ``target_is_slot``: ``target`` is a one-element int64 tensor holding the device address of the
    ``[B, d]`` target, read when the kernel runs (see ``pack_activations_at``); ``x_dtype`` is that
    matrix's element type (float32, bfloat16 or float16)."""
    _need_cuda(target, w_decT, b_dec, b_pre, idx, val, grad_out)
    F, d = w_decT.shape
    B, k = idx.shape
    if det_ws is not None:
        # deterministic accumulation: fixed-point int64 sums in det_ws [F + d + 1] (zeroed by the caller),
        # converted by det_finish; the float atomics on d_b_enc / d_b_dec / stats.sse are not issued
        if det_ws.dtype != torch.int64 or det_ws.numel() < F + d + 1 or not det_ws.is_cuda:
            raise RuntimeError("det_ws must be an int64 CUDA tensor of >= F + d + 1 elements")
    lib = _lib.load()
    if target_is_slot:
        _check_slot(target, "target slot")
        if rows_at is not None:
            _check_slot(rows_at, "rows_at")
        if not w_decT.is_contiguous() or w_decT.dtype != torch.bfloat16:
            raise RuntimeError("w_decT must be contiguous [F, d] bfloat16")
        _run("wsae_decode_backward", lib.wsae_decode_backward_typed, _ptr(target), _ptr(rows_at), _x_dtype_code(x_dtype), _ptr(w_decT), 1, _ptr(b_dec), _ptr(b_pre), _ptr(idx), _ptr(val), _ptr(grad_out), float(coef), B, d, F, k, _ptr(resid), _ptr(resid_bf16), _ptr(stats), _ptr(last_activated), _ptr(step_count), _ptr(d_b_enc), _ptr(d_b_dec), _ptr(dpre_val), _ptr(det_ws), _stream())
    elif det_ws is not None:
        if w_decT.dtype != torch.bfloat16 or not w_decT.is_contiguous():
            raise RuntimeError("w_decT must be contiguous [F, d] bfloat16")
        _run("wsae_decode_backward", lib.wsae_decode_backward_det, _ptr(target), None, _ptr(rows_at), _ptr(w_decT), 1, _ptr(b_dec), _ptr(b_pre), _ptr(idx), _ptr(val), _ptr(grad_out), float(coef), B, d, F, k, _ptr(resid), _ptr(resid_bf16), _ptr(stats), _ptr(last_activated), _ptr(step_count), _ptr(d_b_enc), _ptr(d_b_dec), _ptr(dpre_val), _ptr(det_ws), _stream())
    else:
        _f32c(target, "target")
        if not w_decT.is_contiguous() or w_decT.dtype not in (torch.float32, torch.bfloat16):
            raise RuntimeError("w_decT must be contiguous [F, d] float32 or bfloat16")
        _run("wsae_decode_backward", lib.wsae_decode_backward, _ptr(target), _ptr(w_decT), int(w_decT.dtype == torch.bfloat16), _ptr(b_dec), _ptr(b_pre), _ptr(idx), _ptr(val), _ptr(grad_out), float(coef), B, d, F, k, _ptr(resid), _ptr(resid_bf16), _ptr(stats), _ptr(last_activated), _ptr(step_count), _ptr(d_b_enc), _ptr(d_b_dec), _ptr(dpre_val), _stream())
    if det_ws is not None:
        _run("wsae_det_finish", lib.wsae_det_finish, _ptr(det_ws), F, d, _ptr(grad_out), float(coef), _ptr(d_b_enc), _ptr(d_b_dec), _ptr(stats), _stream())


@dataclass
class TileBuckets:
    """Active (idx, val) entries grouped by (128-feature tile, 64-row chunk) for the K4 GEMMs."""

    offsets: Tensor    # int32 [n_chunks * (n_ft + 1)]
    meta: Tensor       # int32 [B*k]  row_in_chunk | feature_in_tile << 8
    dpre: Tensor       # float32 [B*k]  dv of the entry      (values of the dW_enc GEMM)
    act: Tensor        # float32 [B*k]  relu(val) of the entry (values of the dW_decT GEMM)


def bucket_cells(B: int, F: int) -> tuple[int, int]:
    lib = _lib.load()
    nc, nf = ctypes.c_int(), ctypes.c_int()
    _lib.check(lib.wsae_bucket_cells(B, F, ctypes.byref(nc), ctypes.byref(nf)), "wsae_bucket_cells")
    return nc.value, nf.value


def bucket_supported(F: int, k: int) -> bool:
    """wsae_bucket_by_tile stages one 64-row chunk (64 * k entries of 12 bytes) and the per-tile counts
    in at most 200 KB of shared memory: k <= 256 at every Whisper width.  Larger k: K3's scatter."""
    return (F + 127) // 128 * 4 + 64 * k * 12 <= 200 * 1024


def bucket_by_tile(idx: Tensor, val: Tensor, dpre_val: Tensor, F: int,
                   out: TileBuckets | None = None) -> TileBuckets:
    _need_cuda(idx, val, dpre_val)
    B, k = idx.shape
    n_chunks, n_ft = bucket_cells(B, F)
    dev = idx.device
    if out is None:
        out = TileBuckets(
            torch.empty(n_chunks * (n_ft + 1), dtype=torch.int32, device=dev),
            torch.empty(B * k, dtype=torch.int32, device=dev),
            torch.empty(B * k, dtype=torch.float32, device=dev),
            torch.empty(B * k, dtype=torch.float32, device=dev))
    lib = _lib.load()
    _run("wsae_bucket_by_tile", lib.wsae_bucket_by_tile, _ptr(idx), _ptr(val), _ptr(dpre_val), B, F, k, _ptr(out.offsets), _ptr(out.meta), _ptr(out.dpre), _ptr(out.act), _stream())
    return out


def wgrad_gemm_supported(d: int) -> bool:
    """K4 needs 16-byte aligned bf16 rows for TMA (d % 8 == 0); WSAE_WGRAD=scatter forces K3's
    red.global.add form (kept for the ncu comparison in DESIGN.md)."""
    return d % 8 == 0 and os.environ.get("WSAE_WGRAD", "gemm") != "scatter"


def wgrad_gemm_workspace(B: int, F: int, d: int) -> int:
    """Bytes of split-K workspace the deterministic wgrad GEMM needs at this shape (0 = no split)."""
    lib = _lib.load()
    n = ctypes.c_ulonglong(0)
    _lib.check(lib.wsae_wgrad_gemm_workspace(B, F, d, ctypes.byref(n)), "wsae_wgrad_gemm_workspace")
    return int(n.value)


def wgrad_gemm_(out: Tensor, r_bf16: Tensor, B: int, d: int, buckets: TileBuckets, values: Tensor,
                grad_out: Tensor | None, alpha: float, det_ws: Tensor | None = None) -> None:
    """K4. out[F, d] += alpha * grad_out * S^T @ r_bf16[:B, :d] (S = bucketed sparse entries of the
    same B rows)."""
    _need_cuda(out, r_bf16, values, grad_out)
    _f32c(out, "out")
    if r_bf16.dtype != torch.bfloat16 or r_bf16.dim() != 2 or r_bf16.stride(1) != 1:
        raise RuntimeError("r_bf16 must be a row-major bfloat16 matrix")
    F = out.shape[0]
    if r_bf16.shape[0] < B or r_bf16.shape[1] < d:
        raise RuntimeError("r_bf16 is smaller than [B, d]")
    lib = _lib.load()
    if det_ws is not None:      # ordered split-K reduction through a workspace (bit-reproducible)
        _run("wsae_wgrad_gemm", lib.wsae_wgrad_gemm_det, _ptr(r_bf16), r_bf16.stride(0), B, F, d, _ptr(buckets.offsets), _ptr(buckets.meta), _ptr(values), _ptr(grad_out), float(alpha), _ptr(out), _ptr(det_ws), det_ws.numel() * det_ws.element_size(), _stream(), launches=2)
        return
    _run("wsae_wgrad_gemm", lib.wsae_wgrad_gemm, _ptr(r_bf16), r_bf16.stride(0), B, F, d, _ptr(buckets.offsets), _ptr(buckets.meta), _ptr(values), _ptr(grad_out), float(alpha), _ptr(out), _stream())


def scatter_rows_(out: Tensor, rows: Tensor, center: Tensor | None, idx: Tensor, vals: Tensor) -> None:
    """out[idx[b,j], :] += vals[b,j] * (rows[b,:] - center)  (sparse dW_enc, input width != decoder width)."""
    _need_cuda(out, rows, center, idx, vals)
    _f32c(rows, "rows")
    _f32c(out, "out")
    B, dr = rows.shape
    F = out.shape[0]
    lib = _lib.load()
    _run("wsae_scatter_rows", lib.wsae_scatter_rows, _ptr(rows), _ptr(center), _ptr(idx), _ptr(vals), B, dr, F, idx.shape[1], _ptr(out), _stream())


def bpre_grad(d_b_dec: Tensor, d_b_enc: Tensor, w_enc: Tensor, out: Tensor | None = None,
              det_ws: Tensor | None = None) -> Tensor:
    F, d = w_enc.shape
    if out is None:
        out = torch.empty(d, dtype=torch.float32, device=w_enc.device)
    lib = _lib.load()
    if det_ws is not None:      # fixed summation order: ceil(F / 256) * d floats of workspace
        if det_ws.numel() < (F + 255) // 256 * d:
            raise RuntimeError("bpre_grad det_ws too small")
        _run("wsae_bpre_grad", lib.wsae_bpre_grad_det, _ptr(d_b_dec), _ptr(d_b_enc), _ptr(w_enc), F, d, _ptr(out), _ptr(det_ws), _stream(), launches=2)
        return out
    _run("wsae_bpre_grad", lib.wsae_bpre_grad, _ptr(d_b_dec), _ptr(d_b_enc), _ptr(w_enc), F, d, _ptr(out), _stream())
    return out


def input_grad(resid: Tensor, w_enc: Tensor, idx: Tensor, dpre_val: Tensor,
               grad_out: Tensor | None, coef: float, subtract_g: bool) -> Tensor:
    F, d = w_enc.shape
    B, k = idx.shape
    dx = torch.empty((B, d), dtype=torch.float32, device=resid.device)
    lib = _lib.load()
    _run("wsae_input_grad", lib.wsae_input_grad, _ptr(resid), _ptr(w_enc), _ptr(idx), _ptr(dpre_val), _ptr(grad_out), float(coef), B, d, F, k, int(subtract_g), _ptr(dx), _stream())
    return dx


def renorm_decoder_(w_decT: Tensor, eps: float = 1e-12, shadow: Tensor | None = None) -> None:
    _need_cuda(w_decT, shadow)
    _f32c(w_decT, "w_decT")
    F, d = w_decT.shape
    lib = _lib.load()
    _run("wsae_renorm_decoder", lib.wsae_renorm_decoder, _ptr(w_decT), F, d, eps, _ptr(shadow), _stream())


def counters_update(last_activated: Tensor, step_count: Tensor, threshold: int, bump: bool,
                    dead_count: Tensor | None, *, post: tuple[Tensor | None, Tensor, Tensor] | None = None) -> None:
    """``post = (stats2, seq, mailbox)``: also post {sse, l0 count, dead count, *seq} to ``mailbox``,
    a 4 x int64 PINNED HOST tensor the host polls (``stats2`` / ``seq`` are device int64 tensors)."""
    _need_cuda(last_activated, step_count, dead_count)
    if last_activated.dtype != torch.int64 or step_count.dtype != torch.int64:
        raise RuntimeError("dead-feature counters must be int64")
    lib = _lib.load()
    if post is not None:
        stats2, seq, mailbox = post
        _need_cuda(stats2, seq)
        if mailbox.is_cuda or not mailbox.is_pinned() or mailbox.dtype != torch.int64 or mailbox.numel() < 4:
            raise RuntimeError("mailbox must be a pinned host int64 tensor of >= 4 elements")
        if seq.dtype != torch.int64 or (stats2 is not None and (stats2.dtype != torch.int64 or stats2.numel() < 2)):
            raise RuntimeError("stats2 / seq must be int64 CUDA tensors")
        _run("wsae_counters_update", lib.wsae_counters_update_post, _ptr(last_activated), _ptr(step_count), last_activated.numel(), int(threshold), int(bump), _ptr(dead_count), _ptr(stats2), _ptr(seq), _ptr(mailbox), _stream())
        return
    _run("wsae_counters_update", lib.wsae_counters_update, _ptr(last_activated), _ptr(step_count), last_activated.numel(), int(threshold), int(bump), _ptr(dead_count), _stream())


def densify_hidden(idx: Tensor, val: Tensor, F: int) -> Tensor:
    _need_cuda(idx, val)
    B, k = idx.shape
    hidden = torch.empty((B, F), dtype=torch.float32, device=idx.device)
    lib = _lib.load()
    _run("wsae_densify_hidden", lib.wsae_densify_hidden, _ptr(idx), _ptr(val), B, F, k, _ptr(hidden), _stream())
    return hidden


def cast_bf16(src: Tensor, out: Tensor | None = None) -> Tensor:
    _need_cuda(src)
    _f32c(src, "src")
    if out is None:
        out = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    lib = _lib.load()
    _run("wsae_cast_bf16", lib.wsae_cast_bf16, _ptr(src), _ptr(out), src.numel(), _stream())
    return out


def sumsq_(g: Tensor, out: Tensor, det_ws: Tensor | None = None) -> None:
    """out (float64[1]) += sum(g**2).  ``det_ws`` (float64, >= 1024): ordered, bit-reproducible form."""
    lib = _lib.load()
    if det_ws is not None:
        if det_ws.dtype != torch.float64 or det_ws.numel() < lib.wsae_sumsq_det_blocks():
            raise RuntimeError("sumsq det_ws must be float64 with >= 1024 elements")
        _run("wsae_sumsq", lib.wsae_sumsq_det, _ptr(g), g.numel(), _ptr(det_ws), _ptr(out), _stream(), launches=2)
        return
    _run("wsae_sumsq", lib.wsae_sumsq, _ptr(g), g.numel(), _ptr(out), _stream())


def fused_adamw_(p: Tensor, grad: Tensor, m: Tensor, v: Tensor, hyper: Tensor,
                 grad_sumsq: Tensor | None) -> None:
    lib = _lib.load()
    _run("wsae_fused_adamw", lib.wsae_fused_adamw, _ptr(p), _ptr(grad), _ptr(m), _ptr(v), p.numel(), _ptr(hyper), _ptr(grad_sumsq), _stream())


ADAMW_PROJECT_GRAD = 1     # wsae.h WSAE_ADAMW_PROJECT_GRAD


def adamw_multi_(entries: list[tuple], hyper: Tensor, grad_sumsq: Tensor | None,
                 renorm_eps: float = 1e-12) -> None:
    """Clip + AdamW for several tensors in one launch.  ``entries`` = (param, grad, exp_avg,
    exp_avg_sq, row_len[, flags]): row_len > 0 => rows of that length are re-normalised after the
    update (the feature-major decoder); flags & ADAMW_PROJECT_GRAD => the row gradient is first
    projected off the row direction; all four tensors of an entry share one dense layout."""
    lib = _lib.load()
    arr = (_lib.AdamwTensor * len(entries))()
    for a, ent in zip(arr, entries):
        p, g, m, v, row_len = ent[:5]
        _need_cuda(p, g, m, v)
        a.p, a.g, a.m, a.v = p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr()
        a.n, a.row_len, a.flags = p.numel(), int(row_len), int(ent[5]) if len(ent) > 5 else 0
    _run("wsae_adamw_multi", lib.wsae_adamw_multi, arr, len(entries), _ptr(hyper), _ptr(grad_sumsq), float(renorm_eps), _stream())


def feature_topk_update(feat: Tensor, val: Tensor, rows: Tensor | None, k: int,
                        sample_ids: Tensor | None, sample_base: int, pos_ids: Tensor | None,
                        top_val: Tensor, top_sample: Tensor, top_pos: Tensor, top_count: Tensor,
                        total: Tensor) -> None:
    """Merge a batch of (feature, value) entries into the per-feature top-K lists, in place
    (wsae_feature_topk_update; analysis/feature_viz.py:94-158)."""
    _need_cuda(feat, val, rows, sample_ids, pos_ids, top_val, top_sample, top_pos, top_count, total)
    if feat.dtype != torch.int32 or not feat.is_contiguous():
        raise RuntimeError("feat must be a contiguous int32 tensor")
    _f32c(val, "val")
    _f32c(top_val, "top_val")
    if feat.numel() != val.numel():
        raise RuntimeError("feat and val must have the same number of entries")
    if rows is not None and (rows.dtype != torch.int32 or rows.numel() != feat.numel()):
        raise RuntimeError("rows must be int32 with one entry per (feat, val) pair")
    if sample_ids is not None and sample_ids.dtype != torch.int64:
        raise RuntimeError("sample_ids must be int64")
    if pos_ids is not None and pos_ids.dtype != torch.int32:
        raise RuntimeError("pos_ids must be int32")
    if top_sample.dtype != torch.int64 or top_pos.dtype != torch.int32 or top_count.dtype != torch.int32 \
            or total.dtype != torch.int64:
        raise RuntimeError("tracker state dtypes: top_sample int64, top_pos int32, top_count int32, total int64")
    F, K = top_val.shape
    n = feat.numel()
    if n == 0:
        return
    lib = _lib.load()
    need = ctypes.c_ulonglong(0)
    _lib.check(lib.wsae_feature_topk_workspace(n, F, ctypes.byref(need)), "wsae_feature_topk_workspace")
    ws = torch.empty(need.value, dtype=torch.uint8, device=feat.device)
    _run("wsae_feature_topk_update", lib.wsae_feature_topk_update, _ptr(feat), _ptr(val), _ptr(rows), n,
         int(k), _ptr(sample_ids), int(sample_base), _ptr(pos_ids), F, K, _ptr(top_val), _ptr(top_sample),
         _ptr(top_pos), _ptr(top_count), _ptr(total), _ptr(ws), need.value, _stream(), launches=4)


def layernorm_rows_(x: Tensor, gamma: Tensor | None, beta: Tensor | None, eps: float, out: Tensor,
                    row0: int = 0) -> None:
    """out[row0 : row0 + n, :] = LayerNorm(x.reshape(n, d)) (wsae_layernorm_rows_typed;
    sae/hooks.py:85-86,213-230: final LayerNorm of hooked hidden states + flatten, appended to the
    activation matrix ``out``).  Computed in fp32; ``out`` is float32, bfloat16 or float16, and a half
    ``out`` receives the fp32 result rounded to nearest."""
    _need_cuda(x, gamma, beta, out)
    if x.dtype not in _LN_DTYPES:
        raise RuntimeError(f"unsupported activation dtype {x.dtype}")
    d = x.shape[-1]
    x2 = x.reshape(-1, d)
    if x2.stride(1) != 1:
        x2 = x2.contiguous()
    n = x2.shape[0]
    # a half-precision Whisper carries half-precision LayerNorm parameters: the kernel computes in fp32
    if gamma is not None and gamma.dtype != torch.float32:
        gamma = gamma.to(torch.float32)
    if beta is not None and beta.dtype != torch.float32:
        beta = beta.to(torch.float32)
    _f32c(gamma, "layer_norm.weight")
    _f32c(beta, "layer_norm.bias")
    if out.dtype not in _LN_DTYPES or out.dim() != 2 or out.shape[1] != d or out.stride(1) != 1:
        raise RuntimeError("out must be a float32, bfloat16 or float16 [N, d] matrix with unit column stride")
    if row0 < 0 or row0 + n > out.shape[0]:
        raise RuntimeError(f"rows [{row0}, {row0 + n}) do not fit the [{out.shape[0]}, {d}] activation matrix")
    lib = _lib.load()
    dst = out.data_ptr() + row0 * out.stride(0) * out.element_size()
    _run("wsae_layernorm_rows", lib.wsae_layernorm_rows_typed, _ptr(x2), _LN_DTYPES[x.dtype], n, d, x2.stride(0),
         _ptr(gamma), _ptr(beta), float(eps), dst, _LN_DTYPES[out.dtype], out.stride(0), _stream())


# splice modes of wsae_splice_decode (include/wsae.h)
SPLICE_MODES = {"replace": 0, "error": 1}
SPLICE_MAX_D = 4096


def _splice_rows(h: Tensor, d: int) -> Tensor:
    if h.dtype not in _LN_DTYPES:
        raise RuntimeError(f"unsupported hidden-state dtype {h.dtype} (float32, bfloat16 or float16)")
    if d % 8 != 0 or d > SPLICE_MAX_D:
        raise RuntimeError(f"the splice kernels need d % 8 == 0 and d <= {SPLICE_MAX_D} (got d = {d})")
    h2 = h.reshape(-1, d)
    if not h2.is_contiguous() or h2.data_ptr() % 16 != 0:
        h2 = h2.contiguous()
    return h2


def _ln_params(gamma: Tensor | None, beta: Tensor | None) -> tuple[Tensor | None, Tensor | None]:
    # a half-precision Whisper carries half-precision LayerNorm parameters: the kernels compute in fp32
    gamma = None if gamma is None else gamma.detach().to(torch.float32).contiguous()
    beta = None if beta is None else beta.detach().to(torch.float32).contiguous()
    return gamma, beta


def splice_pack(h: Tensor, gamma: Tensor | None, beta: Tensor | None, eps: float, b_pre: Tensor | None,
                out: Tensor | None = None, row_stats: Tensor | None = None) -> tuple[Tensor, Tensor]:
    """wsae_splice_pack: final LayerNorm of the hidden rows ``h [..., d]`` (float32, bfloat16 or float16)
    and K0's single-term packing in one pass.  Returns (a_packed bf16 [Bp, Kp], row_stats float32 [N, 2] =
    (mean, rstd)); ``a_packed`` equals ``pack_activations(layernorm_rows(h), b_pre, 1)`` bit for bit."""
    _need_cuda(h, gamma, beta, b_pre, out, row_stats)
    d = h.shape[-1]
    h2 = _splice_rows(h, d)
    gamma, beta = _ln_params(gamma, beta)
    _f32c(b_pre, "b_pre")
    N = h2.shape[0]
    if N == 0:
        raise RuntimeError("splice_pack needs at least one row")
    ps = packed_shape(d, 1)
    Bp = _round_up(N, 128)
    if out is None or out.shape != (Bp, ps.kp) or out.dtype != torch.bfloat16:
        out = torch.empty((Bp, ps.kp), dtype=torch.bfloat16, device=h.device)
    if row_stats is None or row_stats.shape != (N, 2):
        row_stats = torch.empty((N, 2), dtype=torch.float32, device=h.device)
    _f32c(row_stats, "row_stats")
    lib = _lib.load()
    _run("wsae_splice_pack", lib.wsae_splice_pack, _ptr(h2), _LN_DTYPES[h2.dtype], N, Bp, d, _ptr(gamma), _ptr(beta),
         float(eps), _ptr(b_pre), _ptr(out), _ptr(row_stats), _stream())
    return out, row_stats


def splice_decode(h: Tensor, row_stats: Tensor | None, gamma: Tensor | None, beta: Tensor | None,
                  w_decT_bf16: Tensor, b_dec: Tensor, b_pre: Tensor | None, idx: Tensor, val: Tensor, *,
                  mode: str, gain: Tensor | None = None, steer: Tensor | None = None, out: Tensor | None = None,
                  stats: Tensor | None = None, x_sum: Tensor | None = None,
                  feature_count: Tensor | None = None) -> Tensor:
    """wsae_splice_decode: the spliced layer output h' (``h``'s shape and dtype) from K1's ``(idx, val)``
    (include/wsae.h states the formulas).  ``row_stats`` from ``splice_pack`` (None: no LayerNorm, x = h).
    ``mode``: "replace" or "error".  Accumulators (caller-zeroed, added to): ``stats`` int64 [3] holding
    {float64 sse, float64 sum x^2, uint64 l0}, ``x_sum`` float64 [d], ``feature_count`` int64 [F]."""
    if mode not in SPLICE_MODES:
        raise RuntimeError(f"unknown splice mode {mode!r} (one of {sorted(SPLICE_MODES)})")
    _need_cuda(h, row_stats, gamma, beta, w_decT_bf16, b_dec, b_pre, idx, val, gain, steer, out, stats, x_sum,
               feature_count)
    F, d = w_decT_bf16.shape
    if h.shape[-1] != d:
        raise RuntimeError(f"hidden width {h.shape[-1]} != decoder width {d}")
    h2 = _splice_rows(h, d)
    N = h2.shape[0]
    if w_decT_bf16.dtype != torch.bfloat16 or not w_decT_bf16.is_contiguous():
        raise RuntimeError("w_decT_bf16 must be a contiguous [F, d] bfloat16 matrix")
    _f32c(b_dec, "decoder.bias")
    _f32c(b_pre, "b_pre")
    _f32c(gain, "gain")
    _f32c(steer, "steer")
    if gain is not None and gain.numel() != F:
        raise RuntimeError(f"gain must have {F} elements")
    if steer is not None and steer.numel() != d:
        raise RuntimeError(f"steer must have {d} elements")
    if idx.dtype != torch.int32 or val.dtype != torch.float32 or idx.shape != val.shape or idx.dim() != 2 \
            or idx.shape[0] != N or not idx.is_contiguous() or not val.is_contiguous():
        raise RuntimeError(f"idx / val must be contiguous int32 / float32 [{N}, k]")
    k = idx.shape[1]
    if row_stats is not None:
        _f32c(row_stats, "row_stats")
        if row_stats.shape != (N, 2):
            raise RuntimeError(f"row_stats must be [{N}, 2]")
        gamma, beta = _ln_params(gamma, beta)
    else:
        gamma = beta = None
    if stats is not None and (stats.dtype != torch.int64 or stats.numel() != 3 or not stats.is_contiguous()):
        raise RuntimeError("stats must be a contiguous int64 [3] tensor")
    if x_sum is not None and (x_sum.dtype != torch.float64 or x_sum.numel() != d or not x_sum.is_contiguous()):
        raise RuntimeError(f"x_sum must be a contiguous float64 [{d}] tensor")
    if feature_count is not None and (feature_count.dtype != torch.int64 or feature_count.numel() != F
                                      or not feature_count.is_contiguous()):
        raise RuntimeError(f"feature_count must be a contiguous int64 [{F}] tensor")
    if out is None:
        out = torch.empty(h.shape, dtype=h.dtype, device=h.device)
    elif out.shape != h.shape or out.dtype != h.dtype or not out.is_contiguous():
        raise RuntimeError("out must be a contiguous tensor of h's shape and dtype")
    if N == 0:
        return out
    lib = _lib.load()
    _run("wsae_splice_decode", lib.wsae_splice_decode, _ptr(h2), _LN_DTYPES[h2.dtype], _ptr(row_stats), _ptr(gamma),
         _ptr(beta), _ptr(w_decT_bf16), _ptr(b_dec), _ptr(b_pre), _ptr(idx), _ptr(val), _ptr(gain), _ptr(steer),
         N, d, F, k, SPLICE_MODES[mode], _ptr(out), _ptr(stats), _ptr(x_sum), _ptr(feature_count), _stream())
    return out
