"""PCB merging (SURVEY.md section 8(f) rank 2); reference: rec_retrieval/merger/algorithms/pcb.py:9-73.

``get_pcb_vectors`` = three exact order statistics per model plus one build pass, all on the GPU:

* the 1 % / 99 % clamp of ``|tau_k|`` (``_clamp(torch.abs(task_vectors), 0.01, 0.01)``, pcb.py:17-27,42) are the
  ``d - int(d*0.01)``-th and ``d - int(d*0.99 - 1)``-th LARGEST magnitudes -- found with the TIES selection kernels;
* the lower clamp of the balancing weights (``_clamp(task_pcb, 1 - density, 0)``, pcb.py:53) is the
  ``int(d*(1-density))``-th smallest of values that only exist on the fly -- ``mr_pcb_vectors`` finds it exactly with a
  sampled key window and ONE pass over the data (three dense histogram passes as the fallback) and never materialises a
  (K, d) temporary.

Floating-point contract: torch's CPU ``exp`` / ``tanh`` and CUDA's differ in the last bit, so the vectors agree with the
reference to ~1e-6 of the row scale except in columns holding an element whose balancing weight lies within a few ulp
of the clamp (there the reference's normalisation is discontinuous: ``scale / max(sum(scale), 1e-12)``)."""
from __future__ import annotations

from typing import List

import torch

from ... import _lib
from ..layout import alloc_rows
from ..types import FlattenedModel
from ._common import as_rows, merge_axpy, weights_tensor
from .ties import select_kth_largest

__all__ = ["get_pcb_vectors", "merge_pcb", "pcb_clamp_ranks"]


def _magnitude_of(cut: torch.Tensor) -> torch.Tensor:
    """fp32 magnitude held in the high word of the selection keys."""
    return (cut >> 32).to(torch.int32).view(torch.float32)


def pcb_clamp_ranks(d: int):
    """(i_lo, i_hi): ascending ranks of the 1 % / 99 % magnitude clamps in a row of d (pcb.py:20-21 with min_ratio =
    max_ratio = 0.01); i_hi wraps like the reference's `sorted_x[-1]` indexing for tiny d."""
    i_lo, i_hi = int(d * 0.01), int(d * (1 - 0.01) - 1)
    return i_lo, (i_hi if i_hi >= 0 else d + i_hi)


def get_pcb_vectors(base_model: FlattenedModel, models: List[FlattenedModel], density: float = 0.2,
                    return_diagnostics: bool = False, force_dense: bool = False, force_ieee: bool = False, **__):
    lib = _lib.load()
    rows = as_rows(models)
    K, d = len(rows), base_model.numel()
    dev = base_model.device
    i_lo, i_hi = pcb_clamp_ranks(d)
    def clamps(defer: bool):
        """1 % / 99 % magnitude clamps (exact order statistics of |tau_k|) and the deferred select statuses."""
        sts = []
        if i_lo == 0:
            # d < 100: sorted_x[0] is the row minimum of |tau| (pcb.py:20); the order-statistic select answers "keep
            # everything" for k = d with cut 0 rather than the d-th largest magnitude, so take the minimum directly
            lo_ = torch.stack([(r - base_model).abs().min() for r in rows]).to(torch.float32).contiguous()
        else:
            c = select_kth_largest(base_model, rows, d - i_lo, defer_status=defer)
            if defer:
                c, st_ = c
                sts.append(st_)
            lo_ = _magnitude_of(c).contiguous()
        c = select_kth_largest(base_model, rows, d - i_hi, defer_status=defer)
        if defer:
            c, st_ = c
            sts.append(st_)
        return lo_, _magnitude_of(c).contiguous(), sts

    q_index = int(d * (1 - density))                             # pcb.py:53: min_ratio = 1 - density, max_ratio = 0
    out = alloc_rows(K, d, dev)
    ldo = max(out.stride(0), d)
    task = alloc_rows(K, d, dev) if return_diagnostics else None
    thr = torch.empty((K, 2), dtype=torch.float32, device=dev) if return_diagnostics else None
    ws_bytes = int(lib.mr_pcb_workspace_bytes(d, K))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    status = torch.zeros(K, dtype=torch.int32, device=dev)

    def run(lo_, hi_, flags: int):
        rc = lib.mr_pcb_vectors(_lib.dptr(base_model, torch.float32), _lib.ptr_array(rows), K, d, _lib.dptr(lo_), _lib.dptr(hi_),
                                q_index, flags, _lib.dptr(status), _lib.dptr(out), ldo, _lib.dptr(task), _lib.dptr(thr),
                                _lib.dptr(ws), ws_bytes, _lib.stream_handle())
        _lib.check(rc, "mr_pcb_vectors")

    # Common case, one host synchronisation for the whole call: both magnitude selects run deferred (sampled bracket),
    # then the fast quantile search (sample, one windowed pass over everything) and the build; the three status words
    # are read together.  A select whose bracket missed is redone on its exact path; a quantile window that missed the
    # wanted rank (status 0) is redone with the three dense radix passes over the whole vector; clamps or ranges outside
    # [2^-60, 2^60] (status 2: the prepared-reciprocal divisions are not valid there) are redone with IEEE divides.
    flags = _lib.MR_PCB_DENSE if force_dense else 0
    if force_ieee:
        flags |= _lib.MR_PCB_IEEE
    lo, hi, sel_status = clamps(defer=True)
    run(lo, hi, flags)
    got = torch.cat(sel_status + [status]).cpu()
    n_sel = sum(int(s.numel()) for s in sel_status)
    if bool((got[:n_sel] != 1).any()):
        lo, hi, _ = clamps(defer=False)
        run(lo, hi, flags)
        got = torch.cat([got[:n_sel], status.cpu()])
    for _ in range(2):          # at most: window missed -> dense, then range -> IEEE (or the other way round)
        st_ = got[n_sel:]
        if bool((st_ == 1).all()):
            break
        if bool((st_ == 0).any()):
            if flags & _lib.MR_PCB_DENSE:
                raise _lib.MergeRecLibraryError("PCB quantile search failed")
            flags |= _lib.MR_PCB_DENSE
        if bool((st_ == 2).any()):
            flags |= _lib.MR_PCB_IEEE
        run(lo, hi, flags)
        got = torch.cat([got[:n_sel], status.cpu()])
    else:
        if bool((got[n_sel:] != 1).any()):
            raise _lib.MergeRecLibraryError(f"PCB vectors failed with status {got[n_sel:].tolist()}")
    if return_diagnostics:
        return out, task, thr, lo, hi
    return out


def merge_pcb(base_model: FlattenedModel, models: List[FlattenedModel], weights: List[float], density: float = 0.2, **__
              ) -> FlattenedModel:
    """``merged = base.clone(); merged += weights[i] * pcb_vector_i`` (pcb.py:61-73): base-first accumulation."""
    assert len(models) == len(weights), "Number of models and weights should match."
    vectors = get_pcb_vectors(base_model, models, density=density)
    return merge_axpy(base_model, list(vectors.unbind(0)), weights_tensor(weights, base_model.device),
                      _lib.MR_ORDER_BASE_FIRST, False)
