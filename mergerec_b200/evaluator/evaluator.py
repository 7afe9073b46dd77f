"""``Evaluator`` -- full-catalog top-K evaluation (reference: rec_retrieval/evaluator/evaluator.py:6-49).

``Evaluator(metrics, ks)(scores, labels, metric_prefix)`` keeps the reference contract (a materialised (Q, N)
score matrix in, ``{prefix}{Recall|NDCG}@{k}`` python floats out, same key order).  Because that contract forces
the caller to build the score matrix (module/recommender/module.py:137, :344-352), two additions take the
embeddings instead and never materialise it: ``topk_embeddings`` and ``evaluate_embeddings`` run the fused
tensor-core scoring + per-row top-K kernel (``mr_score_topk``), shard-aware through ``ShardedItemTable``.

Top-K order is (score desc, item id asc): ``torch.topk``'s order among equal scores is unspecified (SURVEY.md
0.1-D3), so ids can differ from the raw reference only inside groups of exactly equal scores.
"""
from __future__ import annotations

import os
import warnings
from typing import Dict, List, Optional, Tuple, Union

import numpy as np
import torch

from .. import _lib
from .enums import MetricType
from .metrics import label_rank
from .sharded import (MAX_FUSED_TOPK, MR_SCORE_BF16, MR_SCORE_TF32X3, ShardedItemTable, exchange_packed,
                      new_packed_list, split_tf32, to_bf16)

MAX_TOPK = 1024
_warned_item_grad = False


def _warn_item_grad() -> None:
    global _warned_item_grad
    if not _warned_item_grad:
        _warned_item_grad = True
        warnings.warn("label_log_softmax: the item embeddings are a constant of the loss; they receive no gradient",
                      stacklevel=3)
_INT_DTYPES = (torch.int8, torch.int16, torch.int32, torch.int64, torch.uint8)


def exclusion_csr(exclude: torch.Tensor, Q: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """The per-query items to leave out of the ranking -- `exclude`, a (Q, H) integer tensor of global item ids in which
    negative entries are padding (MergeRec pads its sequences with -1) -- as the CSR the kernels take, built with torch
    ops on `exclude`'s device: (offsets int64 (Q + 1), ids int32), row q's ids sorted ascending in
    ids[offsets[q]:offsets[q + 1]].  Duplicates are kept and ids beyond the catalog are allowed (they exclude nothing).
    `ids` has at least one element, so its pointer is valid even when every row is empty."""
    if not isinstance(exclude, torch.Tensor) or exclude.dim() != 2 or exclude.shape[0] != Q:
        raise ValueError(f"exclude must be a (Q, H) tensor with Q = {Q} rows")
    if exclude.dtype not in _INT_DTYPES:
        raise ValueError(f"exclude must hold integer item ids, not {exclude.dtype}")
    x = exclude.to(torch.int64)
    if x.numel() and int(x.max()) >= 1 << 31:
        raise ValueError("exclude holds an item id >= 2^31")
    keep = x >= 0
    counts = keep.sum(dim=1)
    rows = torch.sort(torch.where(keep, x, torch.full_like(x, 1 << 31)), dim=1).values   # padding sorts last
    ids = rows[torch.arange(x.shape[1], device=x.device) < counts[:, None]].to(torch.int32)
    offsets = torch.cat([counts.new_zeros(1), torch.cumsum(counts, dim=0)])
    if ids.numel() == 0:
        ids = torch.zeros(1, dtype=torch.int32, device=x.device)
    return offsets, ids


def _device_csr(exclude: Optional[torch.Tensor], Q: int, dev) -> Optional[Tuple[torch.Tensor, torch.Tensor]]:
    if exclude is None:
        return None
    return tuple(t.to(dev, non_blocking=True) for t in exclusion_csr(exclude, Q))


def _row_chunks(scores: torch.Tensor, dev):
    """(q0, q1, rows q0..q1 of `scores` as fp32 with unit column stride on `dev`): the whole matrix when it is on the
    GPU, otherwise row chunks of at most 1 GiB."""
    Q, N = scores.shape
    rows_per_chunk = Q if scores.is_cuda else max(1, min(Q, (1 << 30) // max(4 * N, 1)))
    for q0 in range(0, Q, max(rows_per_chunk, 1)):
        q1 = min(Q, q0 + rows_per_chunk)
        chunk = scores[q0:q1].to(device=dev, dtype=torch.float32, non_blocking=True)
        yield q0, q1, chunk if chunk.stride(1) == 1 else chunk.contiguous()


def topk_rows(scores: torch.Tensor, k: int, id_base: int = 0,
              exclude: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """(values (Q, k) fp32, ids (Q, k) int32) of a (Q, N) score matrix: `mr_topk_rows`, the drop-in for
    ``torch.topk(scores, k, dim=1)`` (evaluator.py:43).  CPU inputs are copied to the GPU in row chunks.
    `exclude`: (Q, H) global item ids to leave out of each row (negative = padding; `exclusion_csr`), through
    `mr_topk_rows_exclude`; a row left with fewer than k items ends in slots of (-inf, -1)."""
    dev = _lib.require_cuda()
    lib = _lib.load()
    if scores.dim() != 2:
        raise ValueError("scores must be (Q, N)")
    Q, N = scores.shape
    if k > N:
        raise RuntimeError(f"selected index k out of range (k={k}, N={N})")  # torch.topk's error class
    csr = _device_csr(exclude, Q, dev)
    out_v = torch.empty((Q, k), dtype=torch.float32, device=dev)
    out_i = torch.empty((Q, k), dtype=torch.int32, device=dev)
    for q0, q1, chunk in _row_chunks(scores, dev):
        args = (_lib.dptr(chunk), q1 - q0, N, chunk.stride(0), k, id_base, _lib.dptr(out_v[q0:q1]),
                _lib.dptr(out_i[q0:q1]))
        if csr is None:
            _lib.check(lib.mr_topk_rows(*args, _lib.stream_handle()), "mr_topk_rows")
        else:   # the offsets index the whole ids array: the chunk's rows are offsets[q0 : q1 + 1]
            _lib.check(lib.mr_topk_rows_exclude(*args, _lib.dptr(csr[0][q0:]), _lib.dptr(csr[1]), _lib.stream_handle()),
                       "mr_topk_rows_exclude")
    return out_v, out_i


def _own_exclusion(labels: torch.Tensor, exclude: torch.Tensor) -> torch.Tensor:
    """(Q,) bool on the labels' device: label q is in its own `exclude` row."""
    return (exclude.to(device=labels.device, dtype=torch.int64) == labels[:, None]).any(dim=1)


def _exclusion_miss(rank: torch.Tensor, labels: torch.Tensor, exclude: Optional[torch.Tensor]) -> torch.Tensor:
    """The miss rule of every evaluator path: a label inside its own `exclude` row has rank -1."""
    if exclude is None:
        return rank
    return torch.where(_own_exclusion(labels, exclude), torch.full_like(rank, -1), rank)


def _device_labels(labels: torch.Tensor, Q: int, dev) -> torch.Tensor:
    labels = labels.to(device=dev, dtype=torch.int64).contiguous()
    if labels.dim() != 1 or labels.numel() != Q:
        raise ValueError(f"labels must be a (Q,) tensor with Q = {Q}")
    return labels


def rank_rows(scores: torch.Tensor, labels: torch.Tensor, id_base: int = 0,
              exclude: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(Q,) int32 on the GPU: rank[q] = the number of items of row q of a (Q, N) score matrix, minus `exclude[q]`,
    that sort before item labels[q] under the top-K order (score desc, id asc), i.e. the label's 0-based position in
    the full ranking (`mr_rank_rows`); -1 when the label is not an item id of the matrix (id_base + column) or is in
    its own `exclude` row.  CPU inputs are copied to the GPU in row chunks, as in `topk_rows`."""
    dev = _lib.require_cuda()
    lib = _lib.load()
    if scores.dim() != 2:
        raise ValueError("scores must be (Q, N)")
    Q, N = scores.shape
    labels = _device_labels(labels, Q, dev)
    csr = _device_csr(exclude, Q, dev)
    rank = torch.empty(Q, dtype=torch.int32, device=dev)
    for q0, q1, chunk in _row_chunks(scores, dev):
        off, ids = (None, None) if csr is None else (csr[0][q0:], csr[1])   # the offsets index the whole ids array
        _lib.check(lib.mr_rank_rows(_lib.dptr(chunk), q1 - q0, N, chunk.stride(0), id_base, _lib.dptr(labels[q0:q1]),
                                    _lib.dptr(off), _lib.dptr(ids), _lib.dptr(rank[q0:q1]), _lib.stream_handle()),
                   "mr_rank_rows")
    return _exclusion_miss(rank, labels, exclude)


def _workspace(table: ShardedItemTable, query: str, *args) -> Tuple[torch.Tensor, int]:
    """(the table's scratch, its size in bytes) for a call that needs what `lib.<query>(*args)` returns."""
    ws_bytes = int(getattr(_lib.load(), query)(*args))
    if ws_bytes < 0:
        _lib.check(ws_bytes, query)
    return table.workspace(ws_bytes), ws_bytes


def score_topk(user_hi: torch.Tensor, user_lo: Optional[torch.Tensor], table: ShardedItemTable, k: int,
               mode: int = MR_SCORE_TF32X3, out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
               exclude: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Local fused scoring + top-k of pre-split queries against this rank's shard (`mr_score_topk`).  `out` =
    (values (Q, k) fp32, ids (Q, k) int32) to write into (e.g. the planes of the exchange buffer).  `exclude`: (Q, H)
    global item ids to leave out of each row (negative = padding), through `mr_score_topk_exclude`; a row left with
    fewer than k items ends in slots of (-inf, -1)."""
    dev = _lib.require_cuda()
    return _score_topk(user_hi, user_lo, table, k, mode, out, _device_csr(exclude, user_hi.shape[0], dev))


def _score_topk(user_hi, user_lo, table: ShardedItemTable, k: int, mode: int,
                out: Optional[Tuple[torch.Tensor, torch.Tensor]],
                csr: Optional[Tuple[torch.Tensor, torch.Tensor]]) -> Tuple[torch.Tensor, torch.Tensor]:
    """`score_topk` with the exclusion lists already in device CSR form (built once, used for every shard / chunk)."""
    dev = _lib.require_cuda()
    lib = _lib.load()
    Q, E = user_hi.shape
    if E != table.dim:
        raise ValueError(f"embedding dims differ: queries {E}, items {table.dim}")
    if out is None:
        out_v = torch.empty((Q, k), dtype=torch.float32, device=dev)
        out_i = torch.empty((Q, k), dtype=torch.int32, device=dev)
    else:
        out_v, out_i = out
    ws, ws_bytes = _workspace(table, "mr_score_topk_workspace_bytes", Q, table.n_local, E, k)
    args = (_lib.dptr(user_hi), _lib.dptr(user_lo), Q, _lib.dptr(table.hi), _lib.dptr(table.lo), table.n_local, E, k,
            table.id_base, mode, _lib.dptr(out_v), _lib.dptr(out_i), _lib.dptr(ws), ws_bytes)
    if csr is None:
        _lib.check(lib.mr_score_topk(*args, _lib.stream_handle()), "mr_score_topk")
    else:
        _lib.check(lib.mr_score_topk_exclude(*args, _lib.dptr(csr[0]), _lib.dptr(csr[1]), _lib.stream_handle()),
                   "mr_score_topk_exclude")
    return out_v, out_i


def label_score(user_hi: torch.Tensor, user_lo: Optional[torch.Tensor], table: ShardedItemTable, labels: torch.Tensor,
                mode: int = MR_SCORE_TF32X3) -> torch.Tensor:
    """(Q,) int32 holding the uint32 score keys of (query q, item labels[q]) against this rank's shard, bit for bit
    the key of the score `score_topk` ranks, or 0 when this shard does not hold the label (`mr_label_score`).  Over
    the shards of a catalog, the maximum key (unsigned) is the label's key.  `labels`: (Q,) int64 on the device."""
    lib = _lib.load()
    Q, E = user_hi.shape
    key = torch.empty(Q, dtype=torch.int32, device=user_hi.device)
    ws, ws_bytes = _workspace(table, "mr_score_rank_workspace_bytes", Q, table.n_local, E)
    _lib.check(lib.mr_label_score(_lib.dptr(user_hi), _lib.dptr(user_lo), Q, _lib.dptr(table.hi), _lib.dptr(table.lo),
                                  table.n_local, E, table.id_base, mode, _lib.dptr(labels), _lib.dptr(key), _lib.dptr(ws),
                                  ws_bytes, _lib.stream_handle()), "mr_label_score")
    return key


def score_rank(user_hi: torch.Tensor, user_lo: Optional[torch.Tensor], table: ShardedItemTable, labels: torch.Tensor,
               label_key: torch.Tensor, mode: int = MR_SCORE_TF32X3,
               csr: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
               rows: Optional[Tuple[int, int]] = None) -> torch.Tensor:
    """(Q,) int32: the number of this shard's items, minus the row's exclusion list (`csr`, from `exclusion_csr`), that
    sort before the label whose key is `label_key` (`label_score`, maximised over the shards), or -1 where that key is
    0 (`mr_score_rank`).  Over the shards of a catalog the counts add up to the label's rank; the label's own exclusion
    is not applied here.  `rows` = (a, b): count only the shard's local rows [a, b) (a count adds up over any split of
    the catalog, since a score does not depend on where its item sits)."""
    lib = _lib.load()
    Q, E = user_hi.shape
    a, b = (0, table.n_local) if rows is None else rows
    if not 0 <= a <= b <= table.n_local:
        raise ValueError(f"rows [{a}, {b}) outside the shard's {table.n_local} rows")
    hi, lo = table.hi[a:b], None if table.lo is None else table.lo[a:b]
    count = torch.empty(Q, dtype=torch.int32, device=user_hi.device)
    ws, ws_bytes = _workspace(table, "mr_score_rank_workspace_bytes", Q, b - a, E)
    off, ids = (None, None) if csr is None else csr
    _lib.check(lib.mr_score_rank(_lib.dptr(user_hi), _lib.dptr(user_lo), Q, _lib.dptr(hi), _lib.dptr(lo),
                                 b - a, E, table.id_base + a, mode, _lib.dptr(labels), _lib.dptr(label_key),
                                 _lib.dptr(off), _lib.dptr(ids), _lib.dptr(count), _lib.dptr(ws), ws_bytes,
                                 _lib.stream_handle()), "mr_score_rank")
    return count


# Bounded ranks (`label_ranks(cap=...)`): the probe counts the first 1/PROBE_DIV of each shard (whole 256-item tiles);
# the rest of the shard is counted only for the rows whose probe count is still below the cap, gathered into a compact
# query set -- unless more than COMPACT_MAX_LIVE of the rows are live, when the gather would not pay and every row is
# counted in place.  MR_SCORE_PROBE_DIV overrides the probe size (sweeps).
PROBE_DIV = 64
COMPACT_MAX_LIVE = 0.9


def _probe_rows(n_local: int) -> int:
    div = int(os.environ.get("MR_SCORE_PROBE_DIV", "") or PROBE_DIV)
    return min(n_local, 256 * max(1, round(n_local / (256 * max(div, 1)))))


def bounded_count(queries: "PreparedQueries", table: ShardedItemTable, labels: torch.Tensor, key: torch.Tensor,
                  mode: int, csr: Optional[Tuple[torch.Tensor, torch.Tensor]], cap: int) -> torch.Tensor:
    """`score_rank` summed over the catalog's shards where that sum is below `cap`, and some count >= `cap` elsewhere
    (the label's own exclusion not applied; -world on a sharded table where `key` is 0).  A probe over the first
    `_probe_rows` of each shard finishes every row whose count there already reaches `cap`; `mr_rank_compact` /
    `mr_rank_gather` gather the others, the rest of the shard is counted for them alone and added (`mr_rank_add`).
    One host sync (the live count).  On a sharded table: one all-reduce SUM of the Q probe counts, one of the live
    rows' rest counts; every rank gets the same live rows and the same result."""
    lib = _lib.load()
    Q, E = queries.shape
    dev = queries.hi.device
    n_local = table.n_local
    if table.sharded:
        import torch.distributed as dist
    n1 = _probe_rows(n_local)
    count = score_rank(queries.hi, queries.lo, table, labels, key, mode, csr, rows=(0, n1))
    if table.sharded:
        dist.all_reduce(count, op=dist.ReduceOp.SUM, group=table.group)
    elif n1 == n_local:
        return count                    # the probe was the whole table: the counts are exact
    live = torch.empty(1, dtype=torch.int32, device=dev)
    idx = torch.empty(Q, dtype=torch.int32, device=dev)
    labels_c = torch.empty(Q, dtype=torch.int64, device=dev)
    key_c = torch.empty(Q, dtype=torch.int32, device=dev)
    off_c = None if csr is None else torch.empty(Q + 1, dtype=torch.int64, device=dev)
    _lib.check(lib.mr_rank_compact(Q, _lib.dptr(count), cap, _lib.dptr(key), _lib.dptr(labels),
                                   _lib.dptr(None if csr is None else csr[0]), _lib.dptr(live), _lib.dptr(idx),
                                   _lib.dptr(labels_c), _lib.dptr(key_c), _lib.dptr(off_c), _lib.stream_handle()),
               "mr_rank_compact")
    n = int(live.item())
    if n == 0:
        return count
    rows = (n1, n_local)
    in_place = n > COMPACT_MAX_LIVE * Q
    if n1 == n_local:                   # this shard is done; the all-reduce below still needs its (zero) counts
        rest = torch.zeros(Q if in_place else n, dtype=torch.int32, device=dev)
    elif in_place:
        rest = score_rank(queries.hi, queries.lo, table, labels, key, mode, csr, rows=rows)
    else:
        hi = torch.empty((n, E), dtype=queries.hi.dtype, device=dev)
        lo = None if queries.lo is None else torch.empty((n, E), dtype=queries.lo.dtype, device=dev)
        csr_c = None if csr is None else (off_c[:n + 1], torch.empty_like(csr[1]))
        _lib.check(lib.mr_rank_gather(n, _lib.dptr(idx), E * queries.hi.element_size(), _lib.dptr(queries.hi),
                                      _lib.dptr(queries.lo), _lib.dptr(hi), _lib.dptr(lo),
                                      _lib.dptr(None if csr is None else csr[0]), _lib.dptr(None if csr is None else csr[1]),
                                      _lib.dptr(None if csr is None else csr_c[0]),
                                      _lib.dptr(None if csr is None else csr_c[1]), _lib.stream_handle()),
                   "mr_rank_gather")
        rest = score_rank(hi, lo, table, labels_c[:n], key_c[:n], mode, csr_c, rows=rows)
    if table.sharded:
        dist.all_reduce(rest, op=dist.ReduceOp.SUM, group=table.group)
    if in_place:
        idx, n = None, Q
    _lib.check(lib.mr_rank_add(n, _lib.dptr(idx), _lib.dptr(rest), _lib.dptr(count), _lib.stream_handle()),
               "mr_rank_add")
    return count


def score_lse(user_hi: torch.Tensor, user_lo: Optional[torch.Tensor], table: ShardedItemTable, temperature: float,
              mode: int = MR_SCORE_TF32X3, csr: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
              out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """This shard's log-sum-exp partial, (shift (Q,) int32, sum (Q,) fp64): the sum over row q's items, minus its
    exclusion list (`csr`, from `exclusion_csr`), of exp(score / temperature), as sum * 2^shift (`mr_score_lse`).
    `out`: optional (shift, sum) tensors to write into.  `lse_finish` merges the partials of the shards."""
    lib = _lib.load()
    Q, E = user_hi.shape
    if out is None:
        out = (torch.empty(Q, dtype=torch.int32, device=user_hi.device),
               torch.empty(Q, dtype=torch.float64, device=user_hi.device))
    ws, ws_bytes = _workspace(table, "mr_score_lse_workspace_bytes", Q, table.n_local, E)
    off, ids = (None, None) if csr is None else csr
    _lib.check(lib.mr_score_lse(_lib.dptr(user_hi), _lib.dptr(user_lo), Q, _lib.dptr(table.hi), _lib.dptr(table.lo),
                                table.n_local, E, table.id_base, mode, float(temperature), _lib.dptr(off), _lib.dptr(ids),
                                _lib.dptr(out[0]), _lib.dptr(out[1]), _lib.dptr(ws), ws_bytes, _lib.stream_handle()),
               "mr_score_lse")
    return out


def lse_finish(shift: torch.Tensor, sum_: torch.Tensor, label_key: torch.Tensor, temperature: float) -> torch.Tensor:
    """(Q,) fp32: the label's log-softmax over the catalog whose shards' `score_lse` partials are the rows of `shift`
    (P, Q) int32 and `sum_` (P, Q) fp64, merged in row order (`mr_lse_finish`), with `label_key` the label keys of
    `label_score` maximised over the shards; NaN where a key is 0."""
    lib = _lib.load()
    if shift.dim() != 2 or sum_.shape != shift.shape or shift.dtype != torch.int32 or sum_.dtype != torch.float64 \
            or not (shift.is_contiguous() and sum_.is_contiguous()):
        raise ValueError("expected contiguous (P, Q) int32 shifts and (P, Q) float64 sums")
    P, Q = shift.shape
    if label_key.shape != (Q,):
        raise ValueError(f"label_key must be a (Q,) tensor with Q = {Q}")
    logp = torch.empty(Q, dtype=torch.float32, device=shift.device)
    _lib.check(lib.mr_lse_finish(_lib.dptr(shift), _lib.dptr(sum_), P, Q, _lib.dptr(label_key), float(temperature),
                                 _lib.dptr(logp), _lib.stream_handle()), "mr_lse_finish")
    return logp


def score_lse_grad(user_hi: torch.Tensor, user_lo: torch.Tensor, table: ShardedItemTable, temperature: float,
                   labels: torch.Tensor, shift: torch.Tensor, sum_: torch.Tensor, gscale: torch.Tensor,
                   csr: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """This shard's part of the gradient of the label log-softmax with respect to the 3xTF32 queries, (Q, E) fp32:
    -(gscale[q] / temperature) * sum over row q's eligible items n of (p_qn - [n == labels[q]]) * item_n, with p the
    softmax whose normaliser the (P, Q) `score_lse` partials `shift` / `sum_` give (merged as `lse_finish` merges
    them) (`mr_score_lse_grad`).  `out`: optional (Q, E) fp32 tensor the contribution is added to (zeros by default)."""
    lib = _lib.load()
    Q, E = user_hi.shape
    if table.bf16 or user_lo is None:
        raise ValueError("the log-softmax gradient exists for the 3xTF32 operands only")
    if shift.dim() != 2 or sum_.shape != shift.shape or shift.shape[1] != Q or shift.dtype != torch.int32 \
            or sum_.dtype != torch.float64 or not (shift.is_contiguous() and sum_.is_contiguous()):
        raise ValueError(f"expected contiguous (P, {Q}) int32 shifts and (P, {Q}) float64 sums")
    gscale = gscale.to(device=user_hi.device, dtype=torch.float32).contiguous()
    if out is None:
        out = torch.zeros((Q, E), dtype=torch.float32, device=user_hi.device)
    ws, ws_bytes = _workspace(table, "mr_score_lse_grad_workspace_bytes", Q, table.n_local, E)
    off, ids = (None, None) if csr is None else csr
    _lib.check(lib.mr_score_lse_grad(_lib.dptr(user_hi), _lib.dptr(user_lo), Q, _lib.dptr(table.hi), _lib.dptr(table.lo),
                                     table.n_local, E, table.id_base, float(temperature), _lib.dptr(off), _lib.dptr(ids),
                                     _lib.dptr(labels), _lib.dptr(shift), _lib.dptr(sum_), shift.shape[0],
                                     _lib.dptr(gscale), _lib.dptr(out), _lib.dptr(ws), ws_bytes, _lib.stream_handle()),
               "mr_score_lse_grad")
    return out


def _ordered_sum(parts: torch.Tensor) -> torch.Tensor:
    """parts[0] + parts[1] + ... added in index order: the same bits wherever the same (G, ...) stack is summed."""
    total = parts[0].clone()
    for part in parts[1:]:
        total += part
    return total


class _LabelLogSoftmax(torch.autograd.Function):
    """`Evaluator.label_log_softmax` with a backward to the (normalised) query embeddings.  The forward runs the
    kernels of the graph-free call; the backward recomputes the scores chunk by chunk (`score_lse_grad`)."""

    @staticmethod
    def forward(ctx, users, queries, table, labels, temperature, mode, exclude):
        logp, parts = Evaluator._label_log_softmax(queries, table, labels, temperature, mode, exclude)
        ctx.queries, ctx.table, ctx.temperature, ctx.mode = queries, table, temperature, mode
        ctx.labels, ctx.csr, ctx.parts = parts
        ctx.save_for_backward(logp)
        return logp

    @staticmethod
    def backward(ctx, grad_logp):
        if ctx.mode != MR_SCORE_TF32X3:
            raise RuntimeError("label_log_softmax: the gradient exists in MR_SCORE_TF32X3 only; run the forward in "
                               "that mode to train through it")
        (logp,) = ctx.saved_tensors
        queries, table = ctx.queries, ctx.table
        # rows whose label is outside the catalog (NaN) or excluded (-inf) have no gradient
        g = torch.where(logp.isfinite(), grad_logp.to(torch.float32), torch.zeros_like(logp))
        shift, sums = ctx.parts
        dU = score_lse_grad(queries.hi, queries.lo, table, ctx.temperature, ctx.labels, shift, sums, g, ctx.csr)
        if table.sharded:
            # every rank gets the partials of all ranks and adds them in rank order: the same bits on every rank
            import torch.distributed as dist
            gathered = torch.empty((table.world,) + tuple(dU.shape), dtype=dU.dtype, device=dU.device)
            dist.all_gather_into_tensor(gathered.view(-1), dU.view(-1), group=table.group)
            dU = _ordered_sum(gathered)
        return dU, None, None, None, None, None, None


class PreparedQueries:
    """Query embeddings in the operand format of the scoring kernel ((hi, lo) TF32 split, or bf16), prepared once and
    reusable against any number of item tables / evaluations (`Evaluator.prepare_queries`)."""

    def __init__(self, user_emb: torch.Tensor, normalize: bool = False, bf16: bool = False):
        dev = _lib.require_cuda()
        users = user_emb.to(device=dev, dtype=torch.float32)
        if users.dim() != 2:
            raise ValueError("query embeddings must be (Q, E)")
        if normalize:
            users = torch.nn.functional.normalize(users, p=2, dim=-1)   # module/recommender/module.py:74-77
        self.bf16 = bool(bf16)
        self.hi, self.lo = (to_bf16(users), None) if self.bf16 else split_tf32(users)
        self.shape = tuple(users.shape)


class Evaluator:
    def __init__(self, metrics: List[str], ks: List[int]):
        self.metric_names = metrics
        self.ks = ks
        self._max_k = max(ks)
        self._metrics = []
        for metric in metrics:
            for k in ks:
                self._metrics.append(MetricType[metric].metric_cls(k))

    # ------------------------------------------------------------------ reference contract
    def evaluate(self, scores: torch.Tensor, labels: torch.Tensor, metric_prefix: str = "",
                 exclude: Optional[torch.Tensor] = None) -> Dict[str, float]:
        return self(scores, labels, metric_prefix, exclude)

    def __call__(self, scores: torch.Tensor, labels: torch.Tensor, metric_prefix: str = "",
                 exclude: Optional[torch.Tensor] = None) -> Dict[str, float]:
        """`exclude` (optional): (Q, H) global item ids to leave out of each query's ranking (e.g. its history;
        negative entries are padding), as RecBole's full-sort evaluation does.  A label in its row's `exclude`
        cannot be hit: it counts as a miss.  Beyond `topk_rows`'s k <= 1024, the ranks come from `rank_rows`."""
        if self._max_k > MAX_TOPK:
            if self._max_k > scores.shape[-1]:
                raise RuntimeError(f"selected index k out of range (k={self._max_k}, N={scores.shape[-1]})")
            return self.metrics_from_ranks(rank_rows(scores, labels, exclude=exclude), metric_prefix)
        _, ids = topk_rows(scores, self._max_k, exclude=exclude)
        return self.metrics_from_ids(ids, labels, metric_prefix)

    # ------------------------------------------------------------------ fused additions
    def topk_embeddings(self, user_emb: Union[torch.Tensor, PreparedQueries], item_emb: Union[torch.Tensor, ShardedItemTable],
                        k: Optional[int] = None, normalize: bool = False, mode: int = MR_SCORE_TF32X3,
                        exclude: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """Top-k (values fp32, global ids int32), both (Q, k), of ``user_emb @ item_emb.T`` without the matrix.

        ``item_emb`` is an (N, E) tensor (single GPU) or a ``ShardedItemTable`` (reusable, possibly one shard of
        a multi-GPU catalog -- then every rank passes the same queries and receives the same merged lists).
        ``normalize`` applies the reference's cosine normalisation to the queries (and to a raw item tensor).
        ``mode``: ``MR_SCORE_TF32X3`` (default, fp32-faithful), ``MR_SCORE_TF32X1``, or ``MR_SCORE_BF16`` -- the
        bf16-compat mode that mirrors the reference's default ``precision="bf16-mixed"`` runs (bf16 operands, fp32
        accumulation, scores rounded to bf16; configs/base.py:41) with the canonical tie rule on equal scores.
        ``exclude``: (Q, H) global item ids to leave out of each query's list (negative = padding), applied inside the
        fused kernel; a row left with fewer than k items ends in slots of (-inf, -1).  Every rank of a sharded table
        passes the same ``exclude``, like the queries."""
        k = self._max_k if k is None else k
        if k > MAX_FUSED_TOPK:
            raise ValueError(f"fused top-k supports k <= {MAX_FUSED_TOPK}")
        queries, table = self._operands(user_emb, item_emb, normalize, mode, k)
        csr = _device_csr(exclude, queries.shape[0], queries.hi.device)
        if not table.sharded:
            return _score_topk(queries.hi, queries.lo, table, k, mode, None, csr)
        # sharded: the kernel writes this rank's list into the buffer that the single all-gather sends
        local, loc_v, loc_i = new_packed_list(queries.shape[0], k, queries.hi.device)
        _score_topk(queries.hi, queries.lo, table, k, mode, (loc_v, loc_i), csr)
        return exchange_packed(local, k, table.group, gathered=table.gather_buffer(queries.shape[0], k))

    @staticmethod
    def _operands(user_emb, item_emb, normalize: bool, mode: int, k: int) -> Tuple["PreparedQueries", ShardedItemTable]:
        _lib.require_cuda()
        table = item_emb if isinstance(item_emb, ShardedItemTable) else ShardedItemTable(
            item_emb, normalize=normalize, bf16=(mode == MR_SCORE_BF16))
        if table.bf16 != (mode == MR_SCORE_BF16):
            raise ValueError("the item table was prepared for a different scoring mode (bf16 table <-> MR_SCORE_BF16)")
        if k > table.n_total:
            raise RuntimeError(f"selected index k out of range (k={k}, N={table.n_total})")
        queries = user_emb if isinstance(user_emb, PreparedQueries) else PreparedQueries(user_emb, normalize, table.bf16)
        if queries.bf16 != table.bf16:
            raise ValueError("the queries were prepared for a different scoring mode than the item table")
        return queries, table

    def label_ranks(self, user_emb: Union[torch.Tensor, PreparedQueries], item_emb: Union[torch.Tensor, ShardedItemTable],
                    labels: torch.Tensor, normalize: bool = False, mode: int = MR_SCORE_TF32X3,
                    exclude: Optional[torch.Tensor] = None, cap: Optional[int] = None) -> torch.Tensor:
        """(Q,) int32 on the device: rank[q] = the number of items of the whole catalog, minus `exclude[q]`, that sort
        before item labels[q] in query q's ranking (score desc, id asc) -- the label's 0-based position, with no
        ceiling on k.  -1 when the label is not an item id of the catalog or is in its own `exclude` row.  Arguments as
        for `topk_embeddings`.  Computed inside the fused scoring kernel: one pass scores each label (`label_score`),
        one counts the items ahead of it (`score_rank`).  On a sharded table every rank passes the same queries,
        labels and `exclude` and receives the same ranks, after two all-reduces of Q words (MAX of the keys, SUM of
        the counts).

        `cap` (>= 1): a rank is exact where it is below `cap` and is some value >= `cap` elsewhere -- all that Recall@k
        and NDCG@k need for k <= cap.  Rows whose label is already behind `cap` items of a slice of the catalog are not
        scored against the rest of it (`bounded_count`); the ranks below `cap` are the same bits as without it."""
        queries, table = self._operands(user_emb, item_emb, normalize, mode, 1)
        Q = queries.shape[0]
        dev = queries.hi.device
        labels = _device_labels(labels, Q, dev)
        csr = _device_csr(exclude, Q, dev)
        key = self._label_key(queries, table, labels, mode)
        if cap is not None:
            if not 1 <= int(cap) < 1 << 31:
                raise ValueError(f"cap must be in [1, 2^31), not {cap}")
            count = bounded_count(queries, table, labels, key, mode, csr, int(cap))
        else:
            count = score_rank(queries.hi, queries.lo, table, labels, key, mode, csr)
            if table.sharded:
                import torch.distributed as dist
                dist.all_reduce(count, op=dist.ReduceOp.SUM, group=table.group)
        if table.sharded:
            count = torch.where(key == 0, torch.full_like(count, -1), count)
        return _exclusion_miss(count, labels, exclude)

    @staticmethod
    def _label_key(queries: PreparedQueries, table: ShardedItemTable, labels: torch.Tensor, mode: int) -> torch.Tensor:
        """`label_score`; on a sharded table the all-reduce MAX over the ranks, so every rank holds the label's key."""
        key = label_score(queries.hi, queries.lo, table, labels, mode)
        if table.sharded:   # unsigned maximum as a signed one: flip the sign bit
            import torch.distributed as dist
            key ^= -(1 << 31)
            dist.all_reduce(key, op=dist.ReduceOp.MAX, group=table.group)
            key ^= -(1 << 31)
        return key

    @staticmethod
    def label_log_softmax(user_emb: Union[torch.Tensor, PreparedQueries], item_emb: Union[torch.Tensor, ShardedItemTable],
                          labels: torch.Tensor, temperature: float = 1.0, normalize: bool = False,
                          mode: int = MR_SCORE_TF32X3, exclude: Optional[torch.Tensor] = None) -> torch.Tensor:
        """(Q,) fp32 on the device: log_softmax(scores[q] / temperature)[labels[q]] over the whole catalog minus
        `exclude[q]`, without the score matrix -- the per-query log-likelihood of the label, whose negative mean is
        the catalog cross-entropy.  NaN when the label is not an item id of the catalog, -inf when it is in its own
        `exclude` row (probability 0 among the eligible items).  Arguments as for `topk_embeddings`; the scores are
        those the lists rank (bf16-rounded in `MR_SCORE_BF16`).  Computed inside the fused scoring kernel: one pass
        scores each label (`label_score`), one sums exp(score / temperature) per row (`score_lse`).  On a sharded table
        every rank passes the same arguments and receives the same bits, after one all-reduce MAX of the label keys and
        one all-gather of the (shift, sum) partials, merged in rank order (`lse_finish`).

        Differentiable with respect to `user_emb` when it is a tensor that requires grad (through the normalisation
        when `normalize` is set): the backward recomputes the scores in the fused kernel, one catalog chunk at a time,
        and contracts W[q, n] = -(g_q / T) (p_qn - [n == label_q]) with the items without building the (Q, N) matrix
        (`score_lse_grad`).  Rows whose log-probability is NaN or -inf get a zero gradient.  The item embeddings are a
        constant: an item tensor that requires grad gets none (a warning says so once).  `PreparedQueries` are
        constants too.  The backward exists in `MR_SCORE_TF32X3` only; in the other modes it raises.  On a sharded
        table every rank must call backward: each computes its shard's part, one all-gather of the (G, Q, E) parts
        follows, and every rank adds them in rank order, so that all ranks hold the same bits."""
        if isinstance(item_emb, torch.Tensor) and item_emb.requires_grad and torch.is_grad_enabled():
            _warn_item_grad()
            item_emb = item_emb.detach()
        if isinstance(user_emb, torch.Tensor) and user_emb.requires_grad and torch.is_grad_enabled():
            # the torch ops PreparedQueries applies, kept in the graph so that the gradient reaches user_emb
            users = user_emb.to(device=_lib.require_cuda(), dtype=torch.float32)
            if normalize:
                users = torch.nn.functional.normalize(users, p=2, dim=-1)
            queries = PreparedQueries(users.detach(), False, mode == MR_SCORE_BF16)
            queries, table = Evaluator._operands(queries, item_emb, normalize, mode, 1)
            return _LabelLogSoftmax.apply(users, queries, table, labels, temperature, mode, exclude)
        queries, table = Evaluator._operands(user_emb, item_emb, normalize, mode, 1)
        return Evaluator._label_log_softmax(queries, table, labels, temperature, mode, exclude)[0]

    @staticmethod
    def _label_log_softmax(queries: PreparedQueries, table: ShardedItemTable, labels: torch.Tensor, temperature: float,
                           mode: int, exclude: Optional[torch.Tensor]):
        """(logp, (labels, exclusion CSR, (shift, sum) partials of every shard)): the forward of `label_log_softmax`
        and what its backward needs."""
        Q = queries.shape[0]
        dev = queries.hi.device
        labels = _device_labels(labels, Q, dev)
        csr = _device_csr(exclude, Q, dev)
        key = Evaluator._label_key(queries, table, labels, mode)
        if not table.sharded:
            shift, sums = score_lse(queries.hi, queries.lo, table, temperature, mode, csr)
            shift, sums = shift[None], sums[None]
        else:
            # one buffer per rank, (sums fp64 | shifts int32) as 3Q words, written by the kernel and sent by ONE all-gather
            import torch.distributed as dist
            local = torch.empty(3 * Q, dtype=torch.int32, device=dev)
            score_lse(queries.hi, queries.lo, table, temperature, mode, csr,
                      out=(local[2 * Q:], local[:2 * Q].view(torch.float64)))
            gathered = torch.empty((table.world, 3 * Q), dtype=torch.int32, device=dev)
            dist.all_gather_into_tensor(gathered.view(-1), local, group=table.group)
            shift, sums = gathered[:, 2 * Q:].contiguous(), gathered[:, :2 * Q].contiguous().view(torch.float64)
        logp = lse_finish(shift, sums, key, temperature)
        if exclude is not None:   # the miss rule of `_exclusion_miss`, for labels of the catalog
            own = _own_exclusion(labels, exclude) & (key != 0)
            logp = torch.where(own, torch.full_like(logp, -float("inf")), logp)
        return logp, (labels, csr, (shift, sums))

    def topk_embeddings_streamed(self, user_emb: Union[torch.Tensor, "PreparedQueries"], host_items: torch.Tensor,
                                 k: Optional[int] = None, id_base: int = 0, n_total: Optional[int] = None, group=None,
                                 normalize: bool = False, mode: int = MR_SCORE_TF32X3,
                                 first_rows: int = 32768, max_chunks: int = 12,
                                 exclude: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """`topk_embeddings` for an item table that still lives in HOST memory (what `load_item_embeddings` /
        `ItemEncoderMixin.encode_items(...).cpu()` hand over): the rows are copied to the GPU in chunks on a copy stream
        while the previous chunk is being scored, so the transfer hides behind the tensor-core work instead of preceding
        it.  Chunk sizes ramp up geometrically from `first_rows` (only the first, small copy is exposed); every chunk is
        split into its TF32 operands, scored into its own sorted list, and the lists are merged (`mr_topk_merge_packed`).
        Because a (query, item) score does not depend on how the table is cut, the result is bit-identical to the
        one-table call.  `host_items` = this rank's rows (pinned memory makes the copies asynchronous); `id_base`,
        `n_total`, `group` as for `ShardedItemTable`; `exclude` as for `topk_embeddings` (global ids: every chunk
        takes the same lists)."""
        from .sharded import exchange_packed, topk_merge_packed
        k = self._max_k if k is None else k
        if k > MAX_FUSED_TOPK:
            raise ValueError(f"fused top-k supports k <= {MAX_FUSED_TOPK}")
        dev = _lib.require_cuda()
        if host_items.dim() != 2:
            raise ValueError("item table must be (N, E)")
        n_local = int(host_items.shape[0])
        n_total = n_local if n_total is None else int(n_total)
        if k > n_total:
            raise RuntimeError(f"selected index k out of range (k={k}, N={n_total})")
        bf16 = mode == MR_SCORE_BF16
        queries = user_emb if isinstance(user_emb, PreparedQueries) else PreparedQueries(user_emb, normalize, bf16)
        Q = queries.shape[0]
        csr = _device_csr(exclude, Q, dev)
        # chunk plan: geometric ramp, at most max_chunks lists (k * chunks candidates per row must stay mergeable)
        max_chunks = max(1, min(max_chunks, 8192 // max(k, 1)))
        bounds, lo, rows = [], 0, max(int(first_rows), 1)
        while lo < n_local:
            if len(bounds) == max_chunks - 1:
                rows = n_local - lo
            hi = min(n_local, lo + rows)
            bounds.append((lo, hi))
            lo, rows = hi, rows * 2
        C = max(len(bounds), 1)
        partial = torch.empty((C, 2, Q, k), dtype=torch.int32, device=dev)
        if not bounds:        # an empty shard: every list is empty
            partial[:, 0].view(torch.float32).fill_(float("-inf"))
            partial[:, 1].fill_(-1)
        main = torch.cuda.current_stream(dev)
        if not hasattr(self, "_copy_stream"):
            self._copy_stream = torch.cuda.Stream(device=dev)
        copy = self._copy_stream
        copy.wait_stream(main)
        ws = None
        for c, (a, b) in enumerate(bounds):
            with torch.cuda.stream(copy):
                chunk = host_items[a:b].to(device=dev, dtype=torch.float32, non_blocking=True)
                ready = torch.cuda.Event()
                ready.record(copy)
            main.wait_event(ready)
            chunk.record_stream(main)
            table = ShardedItemTable(chunk, id_base=id_base + a, n_total=n_total, normalize=normalize, bf16=bf16)
            table._ws = ws                                            # one scratch for all chunks (grown if needed)
            if b - a >= k:
                _score_topk(queries.hi, queries.lo, table, k, mode, (partial[c, 0].view(torch.float32), partial[c, 1]), csr)
            else:
                self._score_small_chunk(queries, table, k, mode, partial[c], csr)
            ws = table._ws
        vals, ids = topk_merge_packed(partial, k) if C > 1 else (partial[0, 0].view(torch.float32), partial[0, 1])
        if group is not None:
            import torch.distributed as dist
            if dist.get_world_size(group) > 1:
                local = torch.stack([vals.contiguous().view(torch.int32), ids.contiguous()])
                return exchange_packed(local, k, group)
        return vals, ids

    @staticmethod
    def _score_small_chunk(queries: "PreparedQueries", table: ShardedItemTable, k: int, mode: int, out: torch.Tensor,
                           csr: Optional[Tuple[torch.Tensor, torch.Tensor]] = None) -> None:
        """A chunk with fewer than k rows: its list has only n < k entries; the rest of the (Q, k) plane is marked empty."""
        n = table.n_local
        out[0].view(torch.float32).fill_(float("-inf"))
        out[1].fill_(-1)
        if n:
            v, i = _score_topk(queries.hi, queries.lo, table, n, mode, None, csr)
            out[0].view(torch.float32)[:, :n] = v
            out[1][:, :n] = i

    def evaluate_embeddings_streamed(self, user_emb, host_items: torch.Tensor, labels: torch.Tensor, metric_prefix: str = "",
                                     **kw) -> Dict[str, float]:
        """`evaluate_embeddings` with a host-resident item table (see `topk_embeddings_streamed`; `exclude` is one of
        its keywords)."""
        _, ids = self.topk_embeddings_streamed(user_emb, host_items, self._max_k, **kw)
        return self.metrics_from_ids(ids, labels, metric_prefix)

    @staticmethod
    def prepare_queries(user_emb: torch.Tensor, normalize: bool = False, mode: int = MR_SCORE_TF32X3) -> PreparedQueries:
        """Split / convert the query embeddings once; pass the result as `user_emb` to `topk_embeddings` /
        `evaluate_embeddings` as often as needed (several catalogs, several ks, repeated evaluation)."""
        return PreparedQueries(user_emb, normalize, mode == MR_SCORE_BF16)

    def evaluate_embeddings(self, user_emb: Union[torch.Tensor, PreparedQueries], item_emb: Union[torch.Tensor, ShardedItemTable],
                            labels: torch.Tensor, metric_prefix: str = "", normalize: bool = False,
                            mode: int = MR_SCORE_TF32X3, exclude: Optional[torch.Tensor] = None) -> Dict[str, float]:
        """Metrics of `topk_embeddings`; with `exclude`, a label in its row's `exclude` counts as a miss.  The ranks
        come from `label_ranks` with `cap = max(ks)`: a rank at or past max(ks) is a miss for every k, so only the rows
        whose label is still ahead of max(ks) items after a slice of the catalog are scored against the rest of it.
        The floats are those of the top-K lists (`metrics_from_ids(topk_embeddings(...))`), bit for bit."""
        queries, table = self._operands(user_emb, item_emb, normalize, mode, self._max_k)
        return self.metrics_from_ranks(self.label_ranks(queries, table, labels, mode=mode, exclude=exclude,
                                                        cap=self._max_k), metric_prefix)

    # ------------------------------------------------------------------ shared tail
    def metrics_from_ids(self, ids: torch.Tensor, labels: torch.Tensor, metric_prefix: str = "") -> Dict[str, float]:
        """One rank lookup on the GPU (Q int32 back to the host), then every (metric, k) from the same ranks."""
        return self.metrics_from_ranks(label_rank(ids, labels), metric_prefix)

    def metrics_from_ranks(self, ranks: torch.Tensor, metric_prefix: str = "") -> Dict[str, float]:
        """Every (metric, k) from each query's 0-based label rank (-1 = miss), e.g. `label_ranks` or `rank_rows`."""
        ranks = ranks.cpu().numpy() if isinstance(ranks, torch.Tensor) else np.asarray(ranks)
        found = ranks.compress(ranks >= 0)     # compressed once; row order (= the reference's summation order) is kept
        n = int(ranks.shape[0])
        return {metric_prefix + m.name: m.from_found(found, n) for m in self._metrics}
