"""ctypes binding of ``libwsae_sm100.so`` (the C ABI declared in ``include/wsae.h``).

The product path has **no CPU fallback**: if the shared library is missing and cannot be built,
importing the kernels raises; if a kernel call returns non-zero, ``check`` raises ``RuntimeError``.
"""

from __future__ import annotations

import ctypes
import os
import shutil
import subprocess
from ctypes import POINTER, c_double, c_float, c_int, c_int32, c_longlong, c_ulonglong, c_void_p
from pathlib import Path

_PKG = Path(__file__).resolve().parent
# WSAE_LIB_PATH: load another build of the same library (kernel-tuning experiments only)
LIB_PATH = Path(os.environ.get("WSAE_LIB_PATH") or _PKG / "lib" / "libwsae_sm100.so")
CSRC = _PKG / "csrc"

_ERRORS = {
    -1: "WSAE_E_BADARG (bad pointer / shape argument)",
    -2: "WSAE_E_UNSUPPORTED (shape outside the kernel's supported range)",
    -3: "WSAE_E_NODRIVER (cuTensorMapEncodeTiled entry point unavailable)",
}


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile every CUDA source for sm_100a into ``lib/libwsae_sm100.so`` (nvcc cross-compiles)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(nvcc).exists():
        raise RuntimeError("nvcc not found: cannot build libwsae_sm100.so")
    if force:
        subprocess.run(["make", "-C", str(CSRC), "clean"], check=True, capture_output=not verbose)
    proc = subprocess.run(
        ["make", "-C", str(CSRC), "-j", str(os.cpu_count() or 4), f"NVCC={nvcc}"],
        capture_output=True,
        text=True,
    )
    if proc.returncode != 0:
        raise RuntimeError(f"building libwsae_sm100.so failed:\n{proc.stdout}\n{proc.stderr}")
    if verbose:
        print(proc.stdout)
    return LIB_PATH


class AdamwTensor(ctypes.Structure):
    """wsae_adamw_tensor_t (include/wsae.h)."""

    _fields_ = [("p", c_void_p), ("g", c_void_p), ("m", c_void_p), ("v", c_void_p),
                ("n", c_longlong), ("row_len", c_int), ("flags", c_int)]


_SIGNATURES = {
    "wsae_debug_encode_variant": ([c_int], c_int),
    "wsae_debug_encode_mode": ([c_int], c_int),
    "wsae_debug_encode_counters": ([c_void_p], c_int),
    "wsae_debug_wgrad_cluster": ([c_int], c_int),
    "wsae_debug_decode_backward_general": ([c_int], c_int),
    "wsae_adamw_multi": ([POINTER(AdamwTensor), c_int, c_void_p, c_void_p, c_float, c_void_p], c_int),
    "wsae_abi_version": ([], c_int),
    "wsae_packed_k": ([c_int, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int)], c_int),
    "wsae_pack_activations": ([c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p], c_int),
    "wsae_pack_activations_at": ([c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p], c_int),
    "wsae_pack_activations_rows_at": ([c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p], c_int),
    "wsae_pack_activations_typed": ([c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p], c_int),
    "wsae_pack_encoder": ([c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p], c_int),
    "wsae_encode_effective_splits": ([c_int, c_int], c_int),
    "wsae_encode_topk": (
        [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
        c_int,
    ),
    "wsae_encode_topk_dense": (
        [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
         c_void_p, c_void_p, c_void_p, c_void_p],
        c_int,
    ),
    "wsae_encode_topk_chunked": (
        [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
         c_void_p, c_void_p, c_void_p, c_void_p],
        c_int,
    ),
    "wsae_graph_launch": ([c_void_p, c_void_p], c_int),
    "wsae_encode_dense": (
        [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
        c_int,
    ),
    "wsae_row_step": (
        [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
         c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_void_p, c_void_p,
         c_void_p, c_void_p],
        c_int,
    ),
    "wsae_row_step_typed": (
        [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
         c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_void_p, c_void_p,
         c_void_p, c_void_p],
        c_int,
    ),
    "wsae_memcpy_async": ([c_void_p, c_void_p, ctypes.c_size_t, c_void_p], c_int),
    "wsae_decode_mse": (
        [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
         c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
        c_int,
    ),
    "wsae_backward_sparse": (
        [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_float,
         c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p],
        c_int,
    ),
    "wsae_decode_backward": (
        [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
         c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_void_p, c_void_p],
        c_int,
    ),
    "wsae_decode_backward_at": (
        [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
         c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_void_p, c_void_p],
        c_int,
    ),
    "wsae_decode_backward_rows_at": (
        [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
         c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_void_p, c_void_p],
        c_int,
    ),
    "wsae_decode_backward_det": (
        [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
         c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_void_p, c_void_p, c_void_p],
        c_int,
    ),
    "wsae_decode_backward_typed": (
        [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
         c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_void_p, c_void_p, c_void_p],
        c_int,
    ),
    "wsae_det_finish": ([c_void_p, c_int, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p], c_int),
    "wsae_wgrad_gemm_workspace": ([c_int, c_int, c_int, POINTER(c_ulonglong)], c_int),
    "wsae_wgrad_gemm_det": (
        [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
         c_void_p, c_void_p, c_ulonglong, c_void_p],
        c_int,
    ),
    "wsae_sumsq_det_blocks": ([], c_int),
    "wsae_sumsq_det": ([c_void_p, c_longlong, c_void_p, c_void_p, c_void_p], c_int),
    "wsae_bpre_grad_det": ([c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p], c_int),
    "wsae_bucket_cells": ([c_int, c_int, POINTER(c_int), POINTER(c_int)], c_int),
    "wsae_bucket_by_tile": (
        [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p],
        c_int,
    ),
    "wsae_wgrad_gemm": (
        [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
         c_void_p, c_void_p],
        c_int,
    ),
    "wsae_scatter_rows": ([c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p], c_int),
    "wsae_bpre_grad": ([c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p], c_int),
    "wsae_input_grad": (
        [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_int, c_int, c_int, c_int,
         c_int, c_void_p, c_void_p],
        c_int,
    ),
    "wsae_renorm_decoder": ([c_void_p, c_int, c_int, c_float, c_void_p, c_void_p], c_int),
    "wsae_counters_update": ([c_void_p, c_void_p, c_int, c_longlong, c_int, c_void_p, c_void_p], c_int),
    "wsae_counters_update_post": ([c_void_p, c_void_p, c_int, c_longlong, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p], c_int),
    "wsae_densify_hidden": ([c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p], c_int),
    "wsae_cast_bf16": ([c_void_p, c_void_p, c_longlong, c_void_p], c_int),
    "wsae_sumsq": ([c_void_p, c_longlong, c_void_p, c_void_p], c_int),
    "wsae_layernorm_rows": ([c_void_p, c_int, c_longlong, c_int, c_longlong, c_void_p, c_void_p, c_float,
                             c_void_p, c_longlong, c_void_p], c_int),
    "wsae_layernorm_rows_typed": ([c_void_p, c_int, c_longlong, c_int, c_longlong, c_void_p, c_void_p, c_float,
                                   c_void_p, c_int, c_longlong, c_void_p], c_int),
    "wsae_splice_pack": ([c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_void_p, c_void_p,
                          c_void_p, c_void_p], c_int),
    "wsae_splice_decode": (
        [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
        c_int,
    ),
    "wsae_feature_topk_workspace": ([c_longlong, c_int, POINTER(c_ulonglong)], c_int),
    "wsae_feature_topk_update": (
        [c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_void_p, c_longlong, c_void_p, c_int, c_int,
         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_ulonglong, c_void_p],
        c_int,
    ),
    "wsae_fused_adamw": (
        [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_void_p, c_void_p, c_void_p],
        c_int,
    ),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load() -> ctypes.CDLL:
    """Load (building first if necessary) the kernel library. Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        build()
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (argtypes, restype) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == ABI drift; let it propagate loudly
        fn.argtypes = argtypes
        fn.restype = restype
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    if rc in _ERRORS:
        raise RuntimeError(f"{what}: {_ERRORS[rc]}")
    if rc >= 1000:
        raise RuntimeError(f"{what}: cuTensorMapEncodeTiled failed with CUresult {rc - 1000}")
    raise RuntimeError(f"{what}: CUDA error {rc}")
