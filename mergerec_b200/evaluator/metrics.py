"""Recall@k / NDCG@k (reference: rec_retrieval/evaluator/metrics.py:4-88).

The per-row search (`true in pred`, `pred.index(true)`) runs on the GPU as one `mr_label_rank` launch that
returns the position of the label inside each row's predicted list (-1 = absent).  The final reduction is the
reference's own arithmetic, kept on the host so the Python floats come out bit-identical:
`sum(list_of_row_values) / len(list)` in row order, with the NDCG gain `1 / log2_fp32(rank + 2)` taken from a
table built with the very expression the reference evaluates per hit row (metrics.py:84).
"""
from __future__ import annotations

import sys
from typing import List, Optional

import numpy as np
import torch

from .. import _lib


_GAINS = np.zeros(0, dtype=np.float64)


def _gain_table(n: int) -> np.ndarray:
    """gain[r] = 1 / (torch.log2(torch.tensor(r + 2)).item())  -- int64 -> fp32 log2 -> python float -- for r < n.
    One table, extended on demand: each entry costs a torch call, so callers ask only for the ranks that hit."""
    global _GAINS
    if _GAINS.size < n:
        more = [1 / (torch.log2(torch.tensor(r + 2)).item()) for r in range(_GAINS.size, n)]
        _GAINS = np.concatenate([_GAINS, np.asarray(more, dtype=np.float64)])
    return _GAINS[:n]


def _gains(hit_ranks: np.ndarray) -> np.ndarray:
    """The gains of the hit rows' ranks, in row order, from a table only as long as the largest of them needs."""
    if hit_ranks.size == 0:
        return np.zeros(0, dtype=np.float64)
    return np.ascontiguousarray(np.take(_gain_table(int(hit_ranks.max()) + 1), hit_ranks), dtype=np.float64)


def label_rank(ids: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
    """rank[q] = index of labels[q] in ids[q, :], or -1 (int32, on the GPU)."""
    dev = _lib.require_cuda()
    lib = _lib.load()
    ids = ids.to(device=dev, dtype=torch.int32).contiguous()
    labels = labels.to(device=dev, dtype=torch.int64).contiguous()
    if ids.dim() != 2 or labels.dim() != 1 or labels.numel() != ids.shape[0]:
        raise ValueError("expected y_pred (Q, C) and y_true (Q,)")
    Q, K = ids.shape
    rank = torch.empty(Q, dtype=torch.int32, device=dev)
    if Q and K:
        _lib.check(lib.mr_label_rank(_lib.dptr(ids), Q, K, _lib.dptr(labels), _lib.dptr(rank), _lib.stream_handle()),
                   "mr_label_rank")
    elif Q:
        rank.fill_(-1)
    return rank


_SUM_IS_COMPENSATED = sys.version_info >= (3, 12)    # CPython 3.12 switched builtin sum() to Neumaier summation for floats


def _python_float_sum(vals: np.ndarray) -> float:
    """`sum(vals.tolist())` without building the list: `mr_float_sum` replays the interpreter's own float-summation
    loop (compensated on CPython >= 3.12, plain before) on the contiguous float64 array -- the same double, bit for bit
    (asserted against the builtin in the tests), at a few microseconds per 10,000 rows instead of a millisecond."""
    import ctypes as C
    return float(_lib.load().mr_float_sum(C.c_void_p(vals.ctypes.data), int(vals.size), int(_SUM_IS_COMPENSATED)))


def recall_from_ranks(ranks: np.ndarray, k: int) -> float:
    """`sum([1.0 | 0.0 per row]) / len` (metrics.py:49-61).  The sum of n ones is the exact float n, whatever the
    summation order, so the hit count gives the same bits as the reference's row loop."""
    n = int(ranks.shape[0])
    if n == 0:
        return 0.0
    hits = int(np.count_nonzero((ranks >= 0) & (ranks < k)))
    return float(hits) / n if hits else 0 / n


def ndcg_from_ranks(ranks: np.ndarray, k: int) -> float:
    """`sum([gain | 0.0 per row]) / len` in row order (metrics.py:77-88).  The builtin `sum` is kept (CPython >= 3.12
    uses compensated summation for floats, which the reference inherits); rows that miss contribute 0.0, which
    changes neither the running sum nor its compensation term, so only the hit rows are summed -- same bits."""
    n = int(ranks.shape[0])
    if n == 0:
        return 0.0
    hit = (ranks >= 0) & (ranks < k)
    vals = _gains(ranks.compress(hit))
    if vals.size == 0:
        return 0 / n
    return _python_float_sum(vals) / n


def recall_from_found(found: np.ndarray, n: int, k: int) -> float:
    """`recall_from_ranks` on the compressed form: `found` = the ranks of the rows whose label is in the list at all."""
    if n == 0:
        return 0.0
    hits = int(np.count_nonzero(found < k))
    return float(hits) / n if hits else 0 / n


def ndcg_from_found(found: np.ndarray, n: int, k: int) -> float:
    """`ndcg_from_ranks` on the compressed form (row order is preserved by the compression, so the summation order is)."""
    if n == 0:
        return 0.0
    vals = _gains(found.compress(found < k))
    if vals.size == 0:
        return 0 / n
    return _python_float_sum(vals) / n


class BaseMetric:
    METRIC_NAME: Optional[str] = None

    def __init__(self, k: int):
        super().__init__()
        self.k = k

    def __call__(self, y_true: torch.Tensor, y_pred: torch.Tensor) -> float:
        """y_true (Q,) labels, y_pred (Q, C) predicted ids -> metric@k over the first k columns."""
        ranks = label_rank(y_pred[:, : self.k], y_true).cpu().numpy()
        return self.from_ranks(ranks)

    def from_ranks(self, ranks: np.ndarray) -> float:
        raise NotImplementedError("Subclasses must implement this method.")

    def from_found(self, found: np.ndarray, n: int) -> float:
        """Same value from `found = ranks[ranks >= 0]` (computed once for all metrics) and the number of rows."""
        raise NotImplementedError("Subclasses must implement this method.")

    @property
    def name(self) -> str:
        return f"{self.METRIC_NAME}@{self.k}"


class Recall(BaseMetric):
    METRIC_NAME = "Recall"

    def from_ranks(self, ranks: np.ndarray) -> float:
        return recall_from_ranks(ranks, self.k)

    def from_found(self, found: np.ndarray, n: int) -> float:
        return recall_from_found(found, n, self.k)


class NDCG(BaseMetric):
    METRIC_NAME = "NDCG"

    def from_ranks(self, ranks: np.ndarray) -> float:
        return ndcg_from_ranks(ranks, self.k)

    def from_found(self, found: np.ndarray, n: int) -> float:
        return ndcg_from_found(found, n, self.k)
