"""Training-free merges over a flat vector that is SHARDED across GPUs (SURVEY.md section 8(e), merger rows).

The reference is single-process (`ModelMerger`, merger/merger.py:10-107).  Here rank r keeps columns [lo_r, hi_r) of
every flat vector (`flat_shard_bounds`: boundaries are multiples of 32, so ATen's interleaved `torch.sum(dim=0)` order
on the trailing `d mod 32` columns falls entirely on the last rank, exactly where the single-GPU kernels apply it) and:

* task-arithmetic / linear merges need no communication at all (independent columns);
* the TIES trim is GLOBAL over the whole vector (ties.py:14-23), so the k-th largest magnitude is found with three
  radix passes (`mr_ties_mag_hist`) whose (K, 2048) int64 histograms are summed with ONE all-reduce per pass; when
  equal magnitudes straddle the cut, an all-gather of the per-rank tie counts and an exclusive scan in rank order keep
  the lowest GLOBAL indices (the canonical tie rule) -- the result is bit-identical to the single-GPU merge;
* PCB (pcb.py) needs three order statistics per model row -- the 1 % / 99 % magnitude clamps (the sharded select above)
  and the quantile and maximum of the balancing weights (`DistPcb`: the single-GPU search with all-reduced histograms) --
  and is otherwise column-local, so it is bit-identical to the single-GPU merge too;
* DARE is column-local given the keep masks: every rank reads its columns of the (K, d) masks;
* `gather_flat` (one all-gather of the merged slices) rebuilds the full vector where a caller wants it on every rank.

One process per GPU, `torch.distributed` (NCCL over NVLink) for the collectives; with the gloo backend the small
histogram tensors hop through the host, which lets the same code run in world-size-2 tests on one GPU or on CPU
(with `kernels=` replaced by a stand-in -- the product path always uses the CUDA kernels)."""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from .. import _lib
from .algorithms import ties as _ties
from .algorithms._common import as_rows, merge_axpy, weights_tensor
from .algorithms.pcb import _magnitude_of, pcb_clamp_ranks
from .layout import alloc_rows
from .merger import _NEEDS_BASE, ModelMerger
from .types import StateDict
from .utils.model_operations import unflatten_model

__all__ = ["flat_shard_bounds", "sharded_select", "sharded_select_fast", "DistSelect", "get_ties_vectors_sharded", "merge_ties_sharded",
           "merge_task_vector_sharded", "merge_linear_sharded", "DistPcb", "get_pcb_vectors_sharded", "merge_pcb_sharded",
           "merge_dare_sharded", "gather_flat", "ShardedModelMerger", "CudaKernels"]

BINS = 2048


def flat_shard_bounds(d: int, world: int, rank: int) -> Tuple[int, int]:
    """Columns [lo, hi) of the flat vector owned by `rank`: contiguous 32-column blocks, sizes differ by at most one
    block, the (possibly partial) last block goes to the last non-empty rank."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    nblk = (d + 31) // 32
    base, rem = divmod(nblk, world)
    lo_blk = rank * base + min(rank, rem)
    hi_blk = lo_blk + base + (1 if rank < rem else 0)
    return min(lo_blk * 32, d), min(hi_blk * 32, d)


def _world(group) -> Tuple[int, int]:
    if group is None:
        return 1, 0
    import torch.distributed as dist
    return dist.get_world_size(group), dist.get_rank(group)


def _host_hop(t: torch.Tensor, group) -> bool:
    import torch.distributed as dist
    return t.is_cuda and dist.get_backend(group) == "gloo"


def _all_reduce_sum(t: torch.Tensor, group) -> torch.Tensor:
    if group is None:
        return t
    import torch.distributed as dist
    if _host_hop(t, group):
        c = t.cpu()
        dist.all_reduce(c, group=group)
        t.copy_(c)
    else:
        dist.all_reduce(t, group=group)
    return t


def _all_reduce_max(t: torch.Tensor, group) -> torch.Tensor:
    if group is None:
        return t
    import torch.distributed as dist
    if _host_hop(t, group):
        c = t.cpu()
        dist.all_reduce(c, op=dist.ReduceOp.MAX, group=group)
        t.copy_(c)
    else:
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return t


def _all_gather(t: torch.Tensor, group) -> torch.Tensor:
    """(world, *t.shape)."""
    world, _ = _world(group)
    if world == 1:
        return t.unsqueeze(0)
    import torch.distributed as dist
    src = t.cpu() if _host_hop(t, group) else t
    out = torch.empty((world * src.shape[0],) + tuple(src.shape[1:]), dtype=src.dtype, device=src.device)
    dist.all_gather_into_tensor(out, src.contiguous(), group=group)
    return out.view((world,) + tuple(src.shape)).to(t.device)


class CudaKernels:
    """The three kernel entry points the sharded path needs (the product path; tests may inject stand-ins)."""

    @staticmethod
    def rows(models) -> List[torch.Tensor]:
        return as_rows(models)          # raises for anything that is not an fp32 CUDA row: no CPU path

    @staticmethod
    def kth_largest_bits(base, rows, k: int, w):
        """(bit pattern (int64 (K,)) of this slice's k-th largest magnitude, status word) -- the single-GPU selection
        kernels, stream-ordered; the status is checked together with the other flags at the end of the select (a
        failed estimate only widens the search: the windows are verified against the global counts anyway)."""
        cut, status = _ties.select_kth_largest(base, rows, k, w, defer_status=True)
        return cut >> 32, status

    @staticmethod
    def mag_hist(base, rows, w, lo, shift, hist, above, cand=None, cand_count=None) -> None:
        """cand (K, cap, 2) int32 / cand_count (K) int32, optional: (bin, local index) of the in-window elements of
        the models whose shift is 0."""
        d = base.numel()
        rc = _lib.load().mr_ties_mag_hist(_lib.dptr(base, torch.float32), _lib.ptr_array(rows), len(rows), d, _lib.dptr(w),
                                          _lib.dptr(lo, torch.int32), _lib.dptr(shift, torch.int32), _lib.dptr(hist),
                                          _lib.dptr(above), _lib.dptr(cand), _lib.dptr(cand_count),
                                          0 if cand is None else cand.shape[1], _lib.stream_handle())
        _lib.check(rc, "mr_ties_mag_hist")

    @staticmethod
    def ties_build(base, rows, cut, mode: int, w=None, out=None, ldo: int = 0) -> None:
        _ties._build(base, rows, cut, mode, w=w, out=out, ldo=ldo)

    @staticmethod
    def merge(base, rows, w, order: int, src_is_model: bool):
        return merge_axpy(base, rows, w, order, src_is_model)

    @staticmethod
    def alloc_rows(K: int, d: int, device):
        return alloc_rows(K, d, device)


class DistSelect:
    """One rank's side of the stream-ordered sharded select (`mr_ties_select_dist`): the single-GPU sampled-bracket
    algorithm with every counter summed over the ranks and keys that carry GLOBAL indices, so that the cut is the
    single-GPU cut bit for bit.  No host synchronisation and no torch arithmetic between the kernels: per phase one
    library call and one collective on a view of the workspace.

        sel = DistSelect(base_l, rows_l, k_cnt, d_global, lo, w)
        for phase in range(DistSelect.PHASES):
            sel.run(phase, gathered)                      # gathered: only read by the last phase
            if phase < 4:  all-reduce(sel.counters)       # int32 words, sum
            elif phase == 4: gathered = all-gather(sel.survivors)
        sel.cut, sel.status                               # status != 1 somewhere: take the exact path

    `sharded_select` drives it with torch.distributed; tests drive several instances on one GPU by summing the views
    themselves."""

    PHASES = 6

    def __init__(self, base_l: torch.Tensor, rows_l: Sequence[torch.Tensor], k_cnt: int, d_global: int, j_off: int,
                 w: Optional[torch.Tensor] = None):
        import ctypes as C
        lib = _lib.load()
        self.base, self.rows, self.w = base_l, list(rows_l), w
        self.K, self.d_local, self.d_global, self.j_off, self.k_cnt = len(self.rows), base_l.numel(), int(d_global), int(j_off), int(k_cnt)
        dev = base_l.device
        offs = [C.c_int64() for _ in range(4)]
        _lib.check(lib.mr_ties_dist_layout(self.d_local, self.K, *[C.byref(o) for o in offs]), "mr_ties_dist_layout")
        c_off, c_bytes, s_off, s_bytes = (int(o.value) for o in offs)
        self.ws_bytes = int(lib.mr_ties_workspace_bytes(max(self.d_local, 1), self.K)) + 256
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        self.counters = self.ws[c_off:c_off + c_bytes].view(torch.int32)
        self.survivors = self.ws[s_off:s_off + s_bytes]
        self.cut = torch.empty(self.K, dtype=torch.int64, device=dev)
        self.cut_global = torch.empty(self.K, dtype=torch.int64, device=dev)
        self.status = torch.zeros(self.K, dtype=torch.int32, device=dev)
        self._parr = _lib.ptr_array(self.rows) if self.d_local else None

    def run(self, phase: int, gathered: Optional[torch.Tensor] = None, world: int = 1) -> None:
        lib = _lib.load()
        if phase == 5 and gathered is None:
            gathered = self.survivors
        rc = lib.mr_ties_select_dist(_lib.dptr(self.base, torch.float32) if self.d_local else None, self._parr, self.K,
                                     self.d_local, self.j_off, self.d_global, _lib.dptr(self.w), self.k_cnt, phase,
                                     _lib.dptr(gathered), world, _lib.dptr(self.cut), _lib.dptr(self.cut_global),
                                     _lib.dptr(self.status), _lib.dptr(self.ws), self.ws_bytes, _lib.stream_handle())
        _lib.check(rc, "mr_ties_select_dist")


def sharded_select_fast(base_l: torch.Tensor, rows_l: Sequence[torch.Tensor], k_cnt: int, d_global: int, j_off: int,
                        w: Optional[torch.Tensor] = None, group=None):
    """(cut keys for this rank's slice, status) through `DistSelect` and torch.distributed collectives -- six library calls,
    four all-reduces of 33 KB and one all-gather of 262 KB per rank at K = 8, nothing else on the stream, no host sync."""
    world, _ = _world(group)
    sel = DistSelect(base_l, rows_l, k_cnt, d_global, j_off, w)
    gathered = None
    for phase in range(DistSelect.PHASES):
        sel.run(phase, gathered, world)
        if world > 1 and phase < 4:
            _all_reduce_sum(sel.counters, group)
        elif world > 1 and phase == 4:
            import torch.distributed as dist
            gathered = torch.empty(world * sel.survivors.numel(), dtype=torch.uint8, device=base_l.device)
            dist.all_gather_into_tensor(gathered, sel.survivors, group=group)
    return sel.cut, sel.status


def _tie_index(base, row, wk, mag: int, keep: int) -> int:
    """Local index of the `keep`-th (1-based, ascending) element whose weighted-update magnitude has bit pattern `mag`
    (rare path: equal magnitudes straddling the global cut inside this rank)."""
    u = row - base                                   # ties.py:18
    if wk is not None:
        u = u * wk                                   # ties.py:20
    bits = u.view(torch.int32) & 0x7FFFFFFF
    idx = (bits == mag).nonzero().reshape(-1)
    return int(idx[keep - 1])


MARGIN_BITS = 64           # widen the first window by a few bit patterns beyond the per-rank estimates (the proportional
                           # ranks are rounded, so the cut may sit a handful of elements outside their span; a miss is
                           # detected from the counts and falls back to the full range)
FULL_SHIFT = 20            # lo = 0, shift = 20: 2048 bins of 2^20 cover all 31 magnitude bits
CAND_CAP = 1 << 16         # per-model capacity of the (bin, index) list recorded at the last level
TIE_KEEP = 64              # how many of the lowest tied indices are extracted from that list (more: the slice is rescanned)


def _ceil_log2(x: torch.Tensor) -> torch.Tensor:
    """ceil(log2(x)) for int64 x >= 1 (exact: float64 holds 2^31)."""
    return torch.ceil(torch.log2(x.to(torch.float64))).to(torch.int64)


def sharded_select(base_l: torch.Tensor, rows_l: Sequence[torch.Tensor], k_cnt: int, d_global: int,
                   w: Optional[torch.Tensor] = None, group=None, kernels=CudaKernels, defer_status: bool = False,
                   magnitude: bool = False):
    """Per-model cut keys FOR THIS RANK'S SLICE (int64 (K,), bit pattern of the uint64 `mr_ties_build` expects with
    LOCAL indices) such that, over all ranks, exactly the `k_cnt` largest `|w_k (m_k - base)|` of the whole vector
    survive, equal magnitudes resolved towards the lowest global index.

    Product path (`sharded_select_fast` / `mr_ties_select_dist`): the single-GPU sampled-bracket select with all-reduced
    counters, stream-ordered; `defer_status=True` returns `(cut, status)` without any host synchronisation.  If a bracket
    misses (adversarial inputs: millions of equal magnitudes), or with stand-in kernels (CPU tests), the exact windowed
    radix search below runs instead:

    1. every rank takes the proportional order statistic of ITS slice (the single-GPU select, no host sync); the global
       cut lies between the smallest and the largest of them up to the rounding of the ranks, so the first window of
       magnitude bit patterns is their span plus a small margin;
    2. windowed histogram of the slice (`mr_ties_mag_hist`) -> all-reduce -> the window must hold global rank k (else it
       is widened 64-fold, finally to the full range, and the level repeats) -> walk from the top to the bin holding
       rank k -> that bin becomes the next window, 11 bits finer; repeat until a bin is a single bit pattern (one level
       when the shards have the same statistics, up to three for the full range); the last level also records
       (bin, index) of its in-window elements;
    3. all-gather of the per-rank counts AT the cut magnitude, exclusive scan in rank order: lowest global index first.

    `magnitude=True` returns the cut's magnitude bit pattern (int64 (K,), the same on every rank) from the exact search
    instead, without step 3 (the fallback of the PCB clamps after a deferred select reported a miss)."""
    K, dev = len(rows_l), base_l.device
    world, rank = _world(group)
    if k_cnt <= 0:
        return torch.full((K,), -1, dtype=torch.int64, device=dev)          # 0xFFFF...: nothing survives
    if k_cnt >= d_global:
        return torch.zeros(K, dtype=torch.int64, device=dev)                # everything survives
    lo_r, hi_r = flat_shard_bounds(d_global, world, rank)
    if (not magnitude and kernels is CudaKernels and base_l.is_cuda and base_l.numel() == hi_r - lo_r
            and (group is None or not _host_hop(base_l, group))):
        # product path: the stream-ordered device-side select; its status is the only thing the host looks at.  Every
        # rank reaches the same verdict (the brackets are decided from all-reduced counters), so the fallback below is
        # entered by all ranks or by none.
        cut, status = sharded_select_fast(base_l, rows_l, k_cnt, d_global, lo_r, w, group)
        if defer_status:
            return cut, status
        if bool((status.cpu() == 1).all()):
            return cut
    elif defer_status:
        raise _lib.MergeRecLibraryError("defer_status needs the CUDA kernels")
    d_l = base_l.numel()
    if d_l:
        k_l = min(max(int(round(k_cnt * d_l / d_global)), 1), d_l)
        est, est_status = kernels.kth_largest_bits(base_l, rows_l, k_l, w)
        est = est.to(torch.int64).clamp(min=0, max=0x7FFFFFFF)
        if est_status is not None:
            # a slice whose sampled bracket missed has no estimate (like an empty slice): the window then comes from the
            # other ranks, or is the full range
            est = torch.where(est_status.to(est.device) == 1, est, torch.full_like(est, -1))
    else:
        est = torch.full((K,), -1, dtype=torch.int64, device=dev)           # an empty slice has no estimate
    ests = _all_gather(est, group)                                           # (world, K)
    valid = ests >= 0
    big = torch.full_like(ests, 0x7FFFFFFF)
    est_lo = torch.where(valid, ests, big).min(0).values
    est_hi = torch.where(valid, ests, torch.zeros_like(ests)).max(0).values
    margin = MARGIN_BITS

    def window(m):
        lo_ = (est_lo - m).clamp(min=0)
        hi_ = (est_hi + m).clamp(max=0x7FFFFFFF)
        return lo_, (_ceil_log2(hi_ - lo_ + 1) - 11).clamp(min=0)

    lo, shift = window(margin)
    k_t = torch.full((K,), int(k_cnt), dtype=torch.int64, device=dev)
    left = k_t.clone()
    mag = torch.zeros(K, dtype=torch.int64, device=dev)
    mine = torch.zeros(K, dtype=torch.int64, device=dev)
    done = torch.zeros(K, dtype=torch.bool, device=dev)
    n_tie = min(TIE_KEEP, CAND_CAP)
    tie_j = torch.full((K, n_tie), 1 << 40, dtype=torch.int64, device=dev)           # ascending local indices AT the cut
    tie_ok = torch.ones(K, dtype=torch.bool, device=dev)                              # the list was not truncated
    width = torch.full((K,), BINS, dtype=torch.int64, device=dev)    # bins of the current window that belong to the search
    cand = torch.empty((K, CAND_CAP, 2), dtype=torch.int32, device=dev) if d_l else None
    slot = torch.arange(CAND_CAP, device=dev)[None, :]
    bins_idx = torch.arange(BINS, device=dev)[None, :]
    first = True
    for _level in range(12):
        h = torch.zeros((K, BINS), dtype=torch.int64, device=dev)
        a = torch.zeros(K, dtype=torch.int64, device=dev)
        cnt = torch.zeros(K, dtype=torch.int32, device=dev) if d_l else None
        if d_l:
            kernels.mag_hist(base_l, rows_l, w, lo.to(torch.int32), shift.to(torch.int32), h, a, cand, cnt)
        local_hist = h
        both = _all_reduce_sum(torch.cat([h, a[:, None]], dim=1), group)     # (K, BINS + 1): histogram | count above
        hist, above = both[:, :BINS], both[:, BINS]
        if first:
            # the window must contain global rank k_cnt; where it does not (shards with different statistics, rounding of
            # the proportional ranks) widen it 64-fold, finally to the full range, and repeat the level
            miss = (above >= k_t) | (above + hist.sum(1) < k_t)
            if bool(miss.any()):
                margin *= 64
                if margin <= (1 << 18):
                    wlo, wsh = window(margin)
                else:
                    wlo, wsh = torch.zeros_like(lo), torch.full_like(shift, FULL_SHIFT)
                lo, shift = torch.where(miss, wlo, lo), torch.where(miss, wsh, shift)
                continue
            left = k_t - above
            first = False
        # a refined window may be wider than the bin it refines (2048 << shift' >= 1 << shift): ignore the excess bins,
        # their elements were already counted as lying above
        hist = torch.where(bins_idx < width[:, None], hist, torch.zeros_like(hist))
        top = hist.flip(1).cumsum(1)                                         # top[:, i] = count in the i+1 highest bins
        i = (top < left[:, None]).sum(1).clamp(max=BINS - 1)                # first i with top[:, i] >= left
        over = torch.where(i > 0, top.gather(1, (i - 1).clamp(min=0)[:, None]).squeeze(1), torch.zeros_like(left))
        chosen = (BINS - 1) - i
        final = (shift == 0) & ~done
        mag = torch.where(final, lo + chosen, mag)
        mine = torch.where(final, local_hist.gather(1, chosen[:, None]).squeeze(1), mine)
        if cand is not None:
            # local indices of my elements at exactly the cut magnitude, ascending (others pushed to the end)
            n_c = cnt.to(torch.int64).clamp(max=CAND_CAP)
            hit = (slot < n_c[:, None]) & (cand[:, :, 0].to(torch.int64) == chosen[:, None])
            j_all = torch.where(hit, cand[:, :, 1].to(torch.int64) & 0xFFFFFFFF, torch.full_like(hit, 1 << 40, dtype=torch.int64))
            j_low = torch.topk(j_all, n_tie, dim=1, largest=False, sorted=True).values
            tie_j = torch.where(final[:, None], j_low, tie_j)
            tie_ok = torch.where(final, cnt.to(torch.int64) <= CAND_CAP, tie_ok)
        left = torch.where(done, left, left - over)
        lo = torch.where(done, lo, lo + (chosen << shift))
        done = done | final
        new_shift = torch.where(done, torch.zeros_like(shift), (shift - 11).clamp(min=0))
        width = torch.where(done, torch.ones_like(width), (torch.ones_like(shift) << shift) >> new_shift)
        shift = new_shift
        if bool(done.all()):
            break
    else:
        raise _lib.MergeRecLibraryError("sharded TIES select did not converge")
    if magnitude:
        return mag
    counts = _all_gather(mine, group)                                        # (world, K)
    before = counts[:rank].sum(0) if rank > 0 else torch.zeros_like(mine)
    keep = torch.minimum((left - before).clamp(min=0), mine)                 # how many of MY ties survive
    cut_all = mag << 32                                                      # every element at `mag` survives here
    cut_none = (mag + 1) << 32                                               # none does
    cut = torch.where(keep >= mine, cut_all, cut_none)
    partial = (keep > 0) & (keep < mine)
    # the keep-th of my tied elements (ascending local index) is the last survivor: taken from the recorded list ...
    j_keep = tie_j.gather(1, (keep - 1).clamp(min=0, max=n_tie - 1)[:, None]).squeeze(1)
    cut = torch.where(partial, (mag << 32) | (0xFFFFFFFF - j_keep), cut)
    # ... unless that list was truncated or not recorded (millions of equal magnitudes; a first-window miss): rescan
    redo = partial & (~tie_ok | (keep > n_tie) | (j_keep >= (1 << 40)))
    if bool(redo.any()):
        for k in torch.nonzero(redo).reshape(-1).tolist():
            j = _tie_index(base_l, rows_l[k], None if w is None else w.reshape(-1)[k], int(mag[k]), int(keep[k]))
            cut[k] = (int(mag[k]) << 32) | (0xFFFFFFFF - j)
    return cut


def _local(models, kernels) -> List[torch.Tensor]:
    return kernels.rows(models)


def get_ties_vectors_sharded(base_l: torch.Tensor, models_l, density: float, d_global: int, group=None,
                             kernels=CudaKernels) -> torch.Tensor:
    """This rank's columns of `get_ties_vectors` (ties.py:55-72) of the whole vector: (K, d_local)."""
    rows = _local(models_l, kernels)
    K, d = len(rows), base_l.numel()
    cut = sharded_select(base_l, rows, _ties.ties_topk_count(density, d_global), d_global, None, group, kernels)
    out = kernels.alloc_rows(K, d, base_l.device)
    if d:
        kernels.ties_build(base_l, rows, cut, _lib.MR_TIES_VECTORS, out=out, ldo=max(out.stride(0), d))
    return out


def merge_ties_sharded(base_l: torch.Tensor, models_l, weights: Sequence[float], density: float, d_global: int,
                       group=None, kernels=CudaKernels) -> torch.Tensor:
    """This rank's columns of `merge_ties` (ties.py:75-83): weight, global trim, sum -- no election."""
    rows = _local(models_l, kernels)
    assert len(rows) == len(weights), "Number of models and weights should match."
    w = torch.tensor([float(x) for x in weights], dtype=torch.float32, device=base_l.device)
    cut = sharded_select(base_l, rows, _ties.ties_topk_count(density, d_global), d_global, w, group, kernels)
    out = torch.empty_like(base_l)
    if base_l.numel():
        kernels.ties_build(base_l, rows, cut, _lib.MR_TIES_TRIMSUM, w=w, out=out)
    return out


def merge_task_vector_sharded(base_l: torch.Tensor, models_l, weights: Sequence[float], kernels=CudaKernels) -> torch.Tensor:
    """This rank's columns of `merge_task_vector` (task_vector.py:13-34); columns are independent: no collective."""
    rows = _local(models_l, kernels)
    assert len(rows) == len(weights), "Number of models and weights should match."
    if not base_l.numel():
        return torch.empty_like(base_l)
    return kernels.merge(base_l, rows, weights_tensor(weights, base_l.device), _lib.MR_ORDER_BASE_FIRST, True)


def merge_linear_sharded(models_l, weights: Sequence[float], kernels=CudaKernels) -> torch.Tensor:
    """This rank's columns of `merge_linear` (linear.py:8-27)."""
    rows = _local(models_l, kernels)
    assert len(rows) == len(weights), "Number of models and weights should match."
    if not rows[0].numel():
        return torch.empty_like(rows[0])
    return kernels.merge(None, rows, weights_tensor(weights, rows[0].device), _lib.MR_ORDER_LINEAR, False)


class DistPcb:
    """One rank's side of the stream-ordered sharded PCB search (`mr_pcb_vectors_dist`): the single-GPU quantile search of
    `mr_pcb_vectors` (sample, key window, one pass over everything, list refinement; or the three dense passes) with every
    histogram and counter summed over the ranks and the row maxima reduced with MAX, then the build of this rank's
    columns.  No host synchronisation: per phase one library call and up to two all-reduces on views of the workspace.

        pcb = DistPcb(base_l, rows_l, d_global, j_off, flags)
        for phase, coll in enumerate(pcb.collectives):
            pcb.run(phase, clamp_lo, clamp_hi, q_index)
            if coll & MR_PCB_SUM:  all-reduce(sum) of pcb.sum    # int32 words
            if coll & MR_PCB_MAX:  all-reduce(max) of pcb.max    # int32 words
        pcb.out, pcb.status                                      # status as for mr_pcb_vectors, the same on every rank

    `get_pcb_vectors_sharded` drives it with torch.distributed; tests drive several instances on one GPU by reducing the
    views themselves."""

    def __init__(self, base_l: torch.Tensor, rows_l: Sequence[torch.Tensor], d_global: int, j_off: int, flags: int = 0):
        import ctypes as C
        lib = _lib.load()
        self.base, self.rows = base_l, list(rows_l)
        self.K, self.d_local, self.d_global, self.j_off = len(self.rows), base_l.numel(), int(d_global), int(j_off)
        dev = base_l.device
        offs = [C.c_int64() for _ in range(5)]
        _lib.check(lib.mr_pcb_dist_layout(self.d_local, self.d_global, self.K, *[C.byref(o) for o in offs]), "mr_pcb_dist_layout")
        self.ws_bytes, s_off, s_bytes, m_off, m_bytes = (int(o.value) for o in offs)
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        self.sum = self.ws[s_off:s_off + s_bytes].view(torch.int32)
        self.max = self.ws[m_off:m_off + m_bytes].view(torch.int32)
        self.out = alloc_rows(self.K, self.d_local, dev)
        self.status = torch.zeros(self.K, dtype=torch.int32, device=dev)
        self._parr = _lib.ptr_array(self.rows) if self.d_local else None
        self.set_flags(flags)

    def set_flags(self, flags: int) -> None:
        """MR_PCB_DENSE / MR_PCB_IEEE for the next search (the phases and their collectives follow from them)."""
        import ctypes as C
        lib = _lib.load()
        self.flags = int(flags)
        n = lib.mr_pcb_dist_plan(self.d_global, self.flags, None, 0)
        _lib.check(min(n, 0), "mr_pcb_dist_plan")
        plan = (C.c_int32 * n)()
        lib.mr_pcb_dist_plan(self.d_global, self.flags, plan, n)
        self.collectives = [int(c) for c in plan]

    def run(self, phase: int, clamp_lo: torch.Tensor, clamp_hi: torch.Tensor, q_index: int) -> None:
        rc = _lib.load().mr_pcb_vectors_dist(
            _lib.dptr(self.base, torch.float32) if self.d_local else None, self._parr, self.K, self.d_local, self.j_off,
            self.d_global, _lib.dptr(clamp_lo, torch.float32), _lib.dptr(clamp_hi, torch.float32), int(q_index), self.flags,
            phase, _lib.dptr(self.status), _lib.dptr(self.out) if self.d_local else None, max(self.out.stride(0), self.d_local),
            _lib.dptr(self.ws), self.ws_bytes, _lib.stream_handle())
        _lib.check(rc, "mr_pcb_vectors_dist")


def _dist_select_global(base_l, rows_l, k_cnt: int, d_global: int, j_off: int, group):
    """(global cut keys, status) of `DistSelect` with host-hop aware collectives (also over gloo with CUDA tensors)."""
    world, _ = _world(group)
    sel = DistSelect(base_l, rows_l, k_cnt, d_global, j_off)
    gathered = None
    for phase in range(DistSelect.PHASES):
        sel.run(phase, gathered, world)
        if world > 1 and phase < 4:
            _all_reduce_sum(sel.counters, group)
        elif world > 1 and phase == 4:
            gathered = _all_gather(sel.survivors, group).reshape(-1)
    return sel.cut_global, sel.status


def get_pcb_vectors_sharded(base_l: torch.Tensor, models_l, density: float, d_global: int, group=None,
                            force_dense: bool = False, force_ieee: bool = False) -> torch.Tensor:
    """This rank's columns of `get_pcb_vectors` (pcb.py:37-58) of the whole vector, bit for bit: (K, d_local).

    The magnitude clamps are global order statistics of |tau_k| (the sharded select; the row minimum, all-reduced, for
    d_global < 100), the quantile and maximum of the balancing weights come from `DistPcb`, everything else is per
    column.  Like the single-GPU call, the common case synchronises the host once: both selects run deferred, then the
    search and the build; the statuses are reduced over the ranks and read together, and a miss reruns the affected
    step on every rank (exact select; dense passes; IEEE divides)."""
    rows = as_rows(models_l)
    K, d = len(rows), base_l.numel()
    dev = base_l.device
    world, rank = _world(group)
    lo_r, hi_r = flat_shard_bounds(d_global, world, rank)
    if d != hi_r - lo_r:
        raise ValueError(f"rank {rank} holds {d} columns, flat_shard_bounds gives [{lo_r}, {hi_r})")
    i_lo, i_hi = pcb_clamp_ranks(d_global)

    def magnitude(k_cnt: int, defer: bool):
        """fp32 (K,) magnitude of the k_cnt-th largest |tau_k| over the whole vector, and the deferred select status."""
        if k_cnt >= d_global:       # the single-GPU select answers "keep everything" with cut 0
            return torch.zeros(K, dtype=torch.float32, device=dev), None
        if defer:
            cut, st_ = _dist_select_global(base_l, rows, k_cnt, d_global, lo_r, group)
            return _magnitude_of(cut).contiguous(), st_
        mag = sharded_select(base_l, rows, k_cnt, d_global, None, group, magnitude=True)
        return mag.to(torch.int32).view(torch.float32).contiguous(), None

    def clamps(defer: bool):
        sts = []
        if i_lo == 0:
            # d_global < 100: the row minimum of |tau| (pcb.py:20), -max(-x) over the ranks, +inf for an empty slice
            mins = [(r - base_l).abs().min() if d else torch.tensor(float("inf"), device=dev) for r in rows]
            lo_ = _all_reduce_max(-torch.stack(mins).to(torch.float32), group).neg().contiguous()
        else:
            lo_, st_ = magnitude(d_global - i_lo, defer)
            sts.append(st_)
        hi_, st_ = magnitude(d_global - i_hi, defer)
        sts.append(st_)
        return lo_, hi_, [s for s in sts if s is not None]

    q_index = int(d_global * (1 - density))                      # pcb.py:53
    flags = _lib.MR_PCB_DENSE if force_dense else 0
    if force_ieee:
        flags |= _lib.MR_PCB_IEEE
    pcb = DistPcb(base_l, rows, d_global, lo_r, flags)

    def search(lo_, hi_, flags_: int) -> None:
        pcb.set_flags(flags_)
        for phase, coll in enumerate(pcb.collectives):
            pcb.run(phase, lo_, hi_, q_index)
            if world > 1 and coll & _lib.MR_PCB_SUM:
                _all_reduce_sum(pcb.sum, group)
            if world > 1 and coll & _lib.MR_PCB_MAX:
                _all_reduce_max(pcb.max, group)

    def verdict(sel_status):
        """[a select missed, the window missed (status 0), the range needs IEEE divides (status 2)], MAX over the ranks:
        the one host synchronisation of the common case."""
        sel_bad = torch.stack([(s != 1).any() for s in sel_status]).any() if sel_status else torch.zeros((), dtype=torch.bool, device=dev)
        v = torch.stack([sel_bad, (pcb.status == 0).any(), (pcb.status == 2).any()]).to(torch.int32)
        return [bool(x) for x in _all_reduce_max(v, group).cpu()]

    lo, hi, sel_status = clamps(defer=True)
    search(lo, hi, flags)
    sel_bad, miss, rng = verdict(sel_status)
    if sel_bad:
        lo, hi, _ = clamps(defer=False)
        search(lo, hi, flags)
        _, miss, rng = verdict([])
    for _ in range(2):          # at most: window missed -> dense, then range -> IEEE (or the other way round)
        if not (miss or rng):
            break
        if miss:
            if flags & _lib.MR_PCB_DENSE:
                raise _lib.MergeRecLibraryError("PCB quantile search failed")
            flags |= _lib.MR_PCB_DENSE
        if rng:
            flags |= _lib.MR_PCB_IEEE
        search(lo, hi, flags)
        _, miss, rng = verdict([])
    else:
        if miss or rng:
            raise _lib.MergeRecLibraryError(f"PCB vectors failed with status {pcb.status.cpu().tolist()}")
    return pcb.out


def merge_pcb_sharded(base_l: torch.Tensor, models_l, weights: Sequence[float], density: float, d_global: int,
                      group=None) -> torch.Tensor:
    """This rank's columns of `merge_pcb` (pcb.py:61-73): the sharded PCB vectors, then base-first accumulation."""
    assert len(models_l) == len(weights), "Number of models and weights should match."
    vectors = get_pcb_vectors_sharded(base_l, models_l, density, d_global, group)
    if not base_l.numel():
        return torch.empty_like(base_l)
    return merge_axpy(base_l, list(vectors.unbind(0)), weights_tensor(weights, base_l.device), _lib.MR_ORDER_BASE_FIRST, False)


def merge_dare_sharded(base_l: torch.Tensor, models_l, weights: Sequence[float], density: float, d_global: int,
                       masks: Optional[torch.Tensor] = None, generator: Optional[torch.Generator] = None,
                       group=None) -> torch.Tensor:
    """This rank's columns of `merge_dare` (dare.py:9-31), bit for bit.  DARE is column-local given the keep masks:

    * `masks=` (K, d_global), on any device: this rank reads its columns -- in place (leading dimension d_global) when
      the masks are a bool / uint8 tensor on this device, otherwise only its slice is converted and copied;
    * no masks: the whole (K, d_global) mask is drawn from `generator` exactly as `merge_dare` draws it and this rank
      keeps its columns, so equal seeds on every rank give the single-GPU bits.  That costs each rank the transient
      K * d_global * 4 bytes the single-GPU merge pays."""
    assert len(models_l) == len(weights), "Number of models and weights should match."
    p = float(density)
    if p < 0.0 or p > 1.0:
        raise ValueError(f"dropout probability has to be between 0 and 1, but got {p}")
    K, d = len(models_l), base_l.numel()
    if masks is not None and masks.shape != (K, d_global):
        raise ValueError(f"masks must have shape {(K, d_global)}, got {tuple(masks.shape)}")
    rows = as_rows(models_l)
    dev = base_l.device
    world, rank = _world(group)
    lo, hi = flat_shard_bounds(d_global, world, rank)
    if d != hi - lo:
        raise ValueError(f"rank {rank} holds {d} columns, flat_shard_bounds gives [{lo}, {hi})")
    if masks is None:
        masks = torch.empty((K, d_global), dtype=torch.float32, device=dev).bernoulli_(1.0 - p, generator=generator) != 0
    if p == 1.0:                 # torch: `input * zeros`
        keep, scale = torch.zeros((K, d), dtype=torch.uint8, device=dev), 0.0
    elif p == 0.0:               # torch returns the input unchanged
        keep, scale = torch.ones((K, d), dtype=torch.uint8, device=dev), 1.0
    else:
        scale = float(np.float32(1.0) / np.float32(1.0 - p))      # `noise.div_(1 - p)` on an fp32 tensor
        if masks.device == dev and masks.dtype in (torch.bool, torch.uint8) and masks.stride(1) == 1:
            keep = masks.view(torch.uint8)[:, lo:hi]                 # read in place
        else:
            keep = masks[:, lo:hi].to(device=dev).to(torch.uint8).contiguous()
    out = torch.empty_like(base_l)
    if not d:
        return out
    w = weights_tensor(weights, dev)
    rc = _lib.load().mr_merge_dare(_lib.dptr(base_l, torch.float32), _lib.ptr_array(rows), K, d, _lib.dptr(w),
                                   _lib.dptr(keep), keep.stride(0), scale, _lib.dptr(out), _lib.stream_handle())
    _lib.check(rc, "mr_merge_dare")
    return out


def gather_flat(local: torch.Tensor, d_global: int, group=None) -> torch.Tensor:
    """All ranks' slices -> the full flat vector on every rank (one all-gather; slices padded to the largest)."""
    world, rank = _world(group)
    if world == 1:
        return local
    bounds = [flat_shard_bounds(d_global, world, r) for r in range(world)]
    width = max(hi - lo for lo, hi in bounds)
    padded = torch.zeros(width, dtype=local.dtype, device=local.device)
    padded[:local.numel()] = local
    allp = _all_gather(padded, group)
    return torch.cat([allp[r, :hi - lo] for r, (lo, hi) in enumerate(bounds)])


class ShardedModelMerger(ModelMerger):
    """`ModelMerger` (merger/merger.py:10-93) whose flat vectors are sharded over the ranks of `group`.  Same
    constructor and `merge(merge_type, weights, **kwargs)` contract for every merge type ("linear", "task_vector",
    "ties", "pcb", "dare"); the merged state_dict returned on every rank is bit-identical to the single-GPU one.  "dare"
    without `masks=` draws the whole mask from `generator` on every rank (`merge_dare_sharded`): pass generators with
    the same seed on every rank to get the single-GPU bits."""

    def __init__(self, models: Sequence[StateDict], base_model: Optional[StateDict] = None, align_key_order: bool = True,
                 group=None):
        super().__init__(models, base_model, align_key_order)
        self.group = group
        world, rank = _world(group)
        self.d_global = self.models[0].numel()
        lo, hi = flat_shard_bounds(self.d_global, world, rank)
        self.bounds = (lo, hi)
        self.models = [m[lo:hi].clone() for m in self.models]
        if self.base_model is not None:
            self.base_model = self.base_model[lo:hi].clone()

    @torch.no_grad()
    def merge(self, merge_type: str, weights, **kwargs) -> StateDict:
        if isinstance(weights, float):
            weights = [weights] * len(self.models)
        elif not (isinstance(weights, list) and all(isinstance(w, float) for w in weights)):
            raise ValueError("Weights should be a float or a list of floats.")
        if merge_type in _NEEDS_BASE and self.base_model is None:
            raise ValueError(f"{_NEEDS_BASE[merge_type]} merge requires a base model.")
        if merge_type == "linear":
            local = merge_linear_sharded(self.models, weights)
        elif merge_type == "task_vector":
            local = merge_task_vector_sharded(self.base_model, self.models, weights)
        elif merge_type == "ties":
            local = merge_ties_sharded(self.base_model, self.models, weights, kwargs["density"], self.d_global, self.group)
        elif merge_type == "pcb":
            local = merge_pcb_sharded(self.base_model, self.models, weights, kwargs.get("density", 0.2), self.d_global,
                                      self.group)
        elif merge_type == "dare":
            if "density" not in kwargs:       # what ModelMerger's call of merge_dare raises
                raise TypeError("merge_dare() missing 1 required positional argument: 'density'")
            local = merge_dare_sharded(self.base_model, self.models, weights, kwargs["density"], self.d_global,
                                       masks=kwargs.get("masks"), generator=kwargs.get("generator"), group=self.group)
        else:
            raise ValueError(f"Merge type '{merge_type}' is not supported.")
        return unflatten_model(gather_flat(local, self.d_global, self.group), self.shape_dict)
