"""ctypes binding of ``csrc/libmergerec_b200.so`` (C ABI declared in ``include/mergerec_b200.h``).

There is no CPU fallback: if the shared library or a CUDA device is missing, every entry point
raises.  Build with ``python -c "import __graft_entry__ as g; g.build()"`` or ``make -C mergerec_b200/csrc``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libmergerec_b200.so")

MR_ORDER_BASE_FIRST, MR_ORDER_SUM_FIRST, MR_ORDER_LINEAR = 0, 1, 2
MR_TIES_VECTORS, MR_TIES_TRIMSUM, MR_TIES_FUSED_MERGE, MR_TIES_LNS = 0, 1, 2, 3
MR_PCB_DENSE, MR_PCB_IEEE = 1, 2
MR_PCB_SUM, MR_PCB_MAX = 1, 2
MR_MAX_K = 16
MR_DISTILL_MAX_B, MR_DISTILL_MAX_GROUPS, MR_DISTILL_MAX_E = 128, 64, 1024

_lib: Optional[C.CDLL] = None

_vp, _i32, _i64 = C.c_void_p, C.c_int, C.c_int64

# name -> argtypes; must list every function declared in include/mergerec_b200.h
SIGNATURES = {
    "mr_version": ([], C.c_int),
    "mr_last_error": ([], C.c_char_p),
    "mr_task_vectors": ([_vp, _vp, _i32, _i64, _vp, _i64, _vp], C.c_int),
    "mr_merge_axpy": ([_vp, _vp, _i32, _i64, _vp, _i32, _vp, _vp, _i32, _i32, _i32, _vp, _vp], C.c_int),
    "mr_lambda_grad_workspace_bytes": ([_i64, _i32, _i32], _i64),
    "mr_lambda_grad": ([_vp, _vp, _vp, _vp, _i32, _i64, _vp, _i64, _i32, _i32, _vp, _vp, _i64, _vp], C.c_int),
    "mr_ties_workspace_bytes": ([_i64, _i32], _i64),
    "mr_ties_select": ([_vp, _vp, _i32, _i64, _vp, _i64, _vp, _vp, _vp, _i64, _vp], C.c_int),
    "mr_ties_select_exact": ([_vp, _vp, _i32, _i64, _vp, _i64, _vp, _vp, _vp, _i64, _vp], C.c_int),
    "mr_ties_select_build": ([_vp, _vp, _i32, _i64, _i64, _i32, _vp, _i32, _vp, _vp, _i32, _vp, _i64, _vp, _vp, _vp, _i64, _vp], C.c_int),
    "mr_topk_rows": ([_vp, _i64, _i64, _i64, _i32, _i32, _vp, _vp, _vp], C.c_int),
    "mr_topk_rows_exclude": ([_vp, _i64, _i64, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp], C.c_int),
    "mr_topk_merge": ([_vp, _vp, _i32, _i64, _i32, _i32, _vp, _vp, _vp], C.c_int),
    "mr_topk_merge_packed": ([_vp, _i32, _i64, _i32, _i32, _vp, _vp, _vp], C.c_int),
    "mr_float_sum": ([_vp, _i64, _i32], C.c_double),
    "mr_label_rank": ([_vp, _i64, _i32, _vp, _vp, _vp], C.c_int),
    "mr_score_topk_workspace_bytes": ([_i64, _i64, _i32, _i32], _i64),
    "mr_score_topk": ([_vp, _vp, _i64, _vp, _vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _i64, _vp], C.c_int),
    "mr_score_topk_exclude": ([_vp, _vp, _i64, _vp, _vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _i64, _vp, _vp, _vp],
                              C.c_int),
    "mr_score_topk_debug_buffer": ([_vp, _i64], C.c_int),
    "mr_rank_rows": ([_vp, _i64, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp], C.c_int),
    "mr_score_rank_workspace_bytes": ([_i64, _i64, _i32], _i64),
    "mr_label_score": ([_vp, _vp, _i64, _vp, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _i64, _vp], C.c_int),
    "mr_score_rank": ([_vp, _vp, _i64, _vp, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp], C.c_int),
    "mr_score_lse_workspace_bytes": ([_i64, _i64, _i32], _i64),
    "mr_score_lse": ([_vp, _vp, _i64, _vp, _vp, _i64, _i32, _i32, _i32, C.c_float, _vp, _vp, _vp, _vp, _vp, _i64, _vp],
                     C.c_int),
    "mr_lse_finish": ([_vp, _vp, _i64, _i64, _vp, C.c_float, _vp, _vp], C.c_int),
    "mr_score_topk_schedule": ([_i64, _i64, _i32, _i32, _vp, _vp, _i64], _i64),
    "mr_to_bf16": ([_vp, _i64, _vp, _vp], C.c_int),
    "mr_split_tf32": ([_vp, _i64, _vp, _vp, _vp], C.c_int),
    "mr_scores_fp32": ([_vp, _i64, _vp, _i64, _i32, _vp, _i64, _vp], C.c_int),
    "mr_distill_logits": ([_vp, _i32, _i32, _vp, _vp, _i32, _vp, _vp, _i64, _vp], C.c_int),
    "mr_distill_loss": ([_vp, _i64, _vp, _vp, _i32, _i32, C.c_float, C.c_float, C.c_float, _vp, _vp, _i64, _vp], C.c_int),
    "mr_distill_grad_workspace_bytes": ([_i32], _i64),
    "mr_distill_grad": ([_vp, _i64, _vp, _i32, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _i64, _vp], C.c_int),
    "mr_normalize_rows": ([_vp, _i64, _i32, _vp, _vp], C.c_int),
    "mr_pcb_workspace_bytes": ([_i64, _i32], _i64),
    "mr_pcb_vectors": ([_vp, _vp, _i32, _i64, _vp, _vp, _i64, _i32, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp], C.c_int),
    "mr_pcb_dist_layout": ([_i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp], C.c_int),
    "mr_pcb_dist_plan": ([_i64, _i32, _vp, _i32], C.c_int),
    "mr_pcb_vectors_dist": ([_vp, _vp, _i32, _i64, _i64, _i64, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _i64, _vp, _i64, _vp], C.c_int),
    "mr_ties_mag_hist":([_vp, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp], C.c_int),
    "mr_ties_dist_layout": ([_i64, _i32, _vp, _vp, _vp, _vp], C.c_int),
    "mr_ties_select_dist": ([_vp, _vp, _i32, _i64, _i64, _i64, _vp, _i64, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _i64, _vp], C.c_int),
    "mr_merge_dare": ([_vp, _vp, _i32, _i64, _vp, _vp, _i64, C.c_float, _vp, _vp], C.c_int),
    "mr_ties_build": ([_vp, _vp, _i32, _i64, _vp, _i32, _vp, _i32, _vp, _vp, _i32, _vp, _i64, _vp, _vp, _vp], C.c_int),
}


class MergeRecLibraryError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (no CUDA call is made here)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MergeRecLibraryError(
                f"{LIB_PATH} is missing: build it with `make -C {os.path.dirname(LIB_PATH)}` "
                "(there is no CPU fallback for the mergerec_b200 kernels)")
        lib = C.CDLL(LIB_PATH)
        for name, (argtypes, restype) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = argtypes
            fn.restype = restype
        _lib = lib
    return _lib


def require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise MergeRecLibraryError("mergerec_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    msg = load().mr_last_error().decode() or f"status {rc}"
    if rc < 0:
        raise ValueError(f"{what}: {msg}")
    raise MergeRecLibraryError(f"{what}: CUDA error {rc}: {msg}")


def stream_handle() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def dptr(t: Optional[torch.Tensor], dtype: Optional[torch.dtype] = None) -> C.c_void_p:
    """Device pointer of a CUDA tensor (None -> NULL)."""
    if t is None:
        return C.c_void_p(0)
    if not t.is_cuda:
        raise MergeRecLibraryError("expected a CUDA tensor (the kernels have no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"expected {dtype}, got {t.dtype}")
    return C.c_void_p(t.data_ptr())


def ptr_array(tensors: Sequence[torch.Tensor]):
    """Host array of device pointers (the `const float* const*` arguments)."""
    arr = (C.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        if not t.is_cuda or t.dtype != torch.float32:
            raise MergeRecLibraryError("expected fp32 CUDA tensors")
        if t.dim() != 1 or t.stride(0) != 1:
            raise MergeRecLibraryError("expected contiguous 1-D rows")
        arr[i] = t.data_ptr()
    return arr
