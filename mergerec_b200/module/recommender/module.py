"""Evaluation halves of the reference's recommender modules on the fused evaluator kernels
(SURVEY.md section 8(f) row 4; reference: rec_retrieval/module/recommender/module.py).

* ``RecEvaluation``      -- ``RecModule``'s epoch-level evaluation (module.py:284-359): collect the user encodings of a
  whole validation / test epoch, then ONE full-catalog evaluation ``evaluator.evaluate(scores, labels, "val/")`` and the
  cross-entropy over the catalog.  The reference concatenates (num_sequences, num_items) score matrices on the CPU;
  here only the (num_sequences, E) encodings are kept and the score matrix never exists.
* ``RecJointEvaluation`` -- ``RecJointModule``'s per-batch, per-dataloader evaluation (module.py:392-503): every batch of
  dataloader ``i`` is scored against ``item_embeddings[i]`` and evaluated on its own; Lightning then reduces each logged
  key ``{stage}/{metric}/dataloader_idx_{i}`` to a batch-size-weighted mean over the batches (``self.log_dict(...,
  on_epoch=True, batch_size=len(labels))``), and ``on_*_epoch_end`` averages those over the dataloaders with
  ``torch.stack(v).mean()`` (module.py:447-457, 493-503).

Lightning itself is out of scope (and not installable here), so the hooks are plain methods a loop calls and the
logger's reduction is restated: Lightning's mean-reduced ``_ResultMetric`` keeps ``value += metric * batch_size`` and
``cumulated_batch_size += batch_size`` as float32 tensors and returns ``value / cumulated_batch_size``
(lightning/pytorch/trainer/connectors/logger_connector/result.py, ``update`` / ``compute``); parity of that restatement
is UNPINNED (no Lightning to run), the per-batch metric floats themselves are bit-exact (tests).

The encoder forward stays PyTorch; scoring + top-K + Recall / NDCG go through ``Evaluator.evaluate_embeddings``
(``mr_score_topk``: tcgen05 3xTF32 by default, ``MR_SCORE_BF16`` to mirror the reference's bf16-mixed runs), the
catalog cross-entropy through ``Evaluator.label_log_softmax`` in 3xTF32 whatever the metrics' mode, so that the loss
stays the fp32 cross-entropy of the reference.
"""
from __future__ import annotations

from collections import defaultdict
from typing import Dict, List, Literal, Optional, Sequence, Union

import torch
from torch import nn

from ...evaluator import Evaluator, ShardedItemTable
from ...evaluator.evaluator import PreparedQueries
from ...evaluator.sharded import MR_SCORE_BF16, MR_SCORE_TF32X3

__all__ = ["RecEvaluation", "RecJointEvaluation", "WeightedMeanLog", "catalog_cross_entropy"]


def catalog_cross_entropy(user_encoding: Union[torch.Tensor, PreparedQueries],
                          item_embeddings: Union[torch.Tensor, ShardedItemTable], labels: torch.Tensor,
                          temperature: float) -> torch.Tensor:
    """``nn.functional.cross_entropy(scores / temperature, labels)`` with ``scores = user @ items.T`` (module.py:307, :363),
    as ``-Evaluator.label_log_softmax(...).mean()`` in 3xTF32: the fused scoring kernel, no logits in memory.  The mean is
    taken in fp64 and returned as a 0-d fp32 tensor on the device.  The operands may also be prepared for 3xTF32
    (``PreparedQueries`` / a ``ShardedItemTable`` without bf16).  Labels outside ``[0, num_items)`` raise ``ValueError``."""
    n_items = item_embeddings.n_total if isinstance(item_embeddings, ShardedItemTable) else int(item_embeddings.shape[0])
    if labels.numel() and not bool(((labels >= 0) & (labels < n_items)).all()):
        raise ValueError(f"labels must be item ids in [0, {n_items})")
    logp = Evaluator.label_log_softmax(user_encoding, item_embeddings, labels, temperature, mode=MR_SCORE_TF32X3)
    return (-logp.to(torch.float64).sum() / max(logp.shape[0], 1)).to(torch.float32)


class WeightedMeanLog:
    """Lightning's epoch reduction of ``self.log(key, value, on_epoch=True, batch_size=n)`` restated: per key a float32
    running ``value += v * n`` and ``cumulated_batch_size += n``; ``compute()`` = ``value / cumulated_batch_size``."""

    def __init__(self):
        self._value: Dict[str, torch.Tensor] = {}
        self._count: Dict[str, torch.Tensor] = {}

    def log(self, key: str, value: Union[float, torch.Tensor], batch_size: int) -> None:
        v = torch.as_tensor(value).detach().to(device="cpu", dtype=torch.float32)
        if key not in self._value:
            self._value[key] = torch.zeros((), dtype=torch.float32)
            self._count[key] = torch.zeros((), dtype=torch.float32)
        self._value[key] = self._value[key] + v * batch_size
        self._count[key] = self._count[key] + batch_size

    def log_dict(self, metrics: Dict[str, Union[float, torch.Tensor]], batch_size: int) -> None:
        for k, v in metrics.items():
            self.log(k, v, batch_size)

    def compute(self) -> Dict[str, torch.Tensor]:
        return {k: self._value[k] / self._count[k] for k in self._value}


class _EvalBase:
    def __init__(self, evaluator: Evaluator, similarity: Literal["dot", "cosine"], temperature: float = 0.05,
                 mode: int = MR_SCORE_TF32X3):
        self.evaluator = evaluator
        self.similarity = similarity
        self.temperature = temperature
        self.mode = mode

    def _maybe_normalize(self, matrix: torch.Tensor) -> torch.Tensor:
        if self.similarity == "cosine":
            return nn.functional.normalize(matrix, p=2, dim=-1)    # module.py:74-77
        return matrix

    def _table(self, items: Union[torch.Tensor, ShardedItemTable]) -> ShardedItemTable:
        if isinstance(items, ShardedItemTable):
            return items
        return ShardedItemTable(items.detach(), bf16=(self.mode == MR_SCORE_BF16))

    @staticmethod
    def _loss_table(items: torch.Tensor, table: ShardedItemTable) -> ShardedItemTable:
        """The 3xTF32 operand of the loss: the metric table itself, or a TF32-split table when that one is bf16."""
        return ShardedItemTable(items.detach()) if table.bf16 else table

    @staticmethod
    def _queries(users: torch.Tensor, table: ShardedItemTable) -> Union[torch.Tensor, PreparedQueries]:
        """Queries prepared once for the metrics and the loss when both take the TF32 split, else left raw."""
        return users if table.bf16 else PreparedQueries(users)


class RecEvaluation(_EvalBase):
    """``RecModule``'s validation / test epoch (module.py:284-359) without the score matrices."""

    def __init__(self, evaluator: Evaluator, similarity: Literal["dot", "cosine"], temperature: float = 0.05,
                 mode: int = MR_SCORE_TF32X3):
        super().__init__(evaluator, similarity, temperature, mode)
        self.item_embeddings: Optional[torch.Tensor] = None      # injected like ItemEncodingCallback does
        self._table_cache: Optional[ShardedItemTable] = None
        self._loss_table_cache: Optional[ShardedItemTable] = None
        self.eval_user_embeddings: List[torch.Tensor] = []
        self.eval_labels: List[torch.Tensor] = []

    def set_item_embeddings(self, item_embeddings: torch.Tensor) -> None:
        self.item_embeddings = item_embeddings
        self._table_cache = None
        self._loss_table_cache = None

    def on_epoch_start(self) -> None:
        self.eval_user_embeddings, self.eval_labels = [], []

    def step(self, user_encoding: torch.Tensor, labels: torch.Tensor) -> None:
        """One batch: keep the (normalised) user encodings and labels (the reference keeps the scores, module.py:304-305)."""
        self.eval_user_embeddings.append(self._maybe_normalize(user_encoding.detach()).to(torch.float32))
        self.eval_labels.append(labels.detach())

    def on_epoch_end(self, stage: str = "val") -> Dict[str, float]:
        """module.py:311-323 / :345-359: one full-catalog evaluation of the whole epoch + the epoch loss."""
        if self.item_embeddings is None:
            raise RuntimeError("item_embeddings have not been injected")
        users = torch.cat(self.eval_user_embeddings, dim=0)
        labels = torch.cat(self.eval_labels, dim=0)
        if self._table_cache is None:
            self._table_cache = self._table(self.item_embeddings)
            self._loss_table_cache = self._loss_table(self.item_embeddings, self._table_cache)
        queries = self._queries(users, self._table_cache)
        metrics = self.evaluator.evaluate_embeddings(queries, self._table_cache, labels, metric_prefix=f"{stage}/", mode=self.mode)
        loss = catalog_cross_entropy(queries, self._loss_table_cache, labels, self.temperature)
        metrics[f"{stage}/epoch_loss" if stage == "val" else f"{stage}/loss"] = loss.item()
        return metrics


class RecJointEvaluation(_EvalBase):
    """``RecJointModule``'s per-batch evaluation over several dataloaders (module.py:392-503)."""

    def __init__(self, evaluator: Evaluator, similarity: Literal["dot", "cosine"], temperature: float = 0.05,
                 mode: int = MR_SCORE_TF32X3):
        super().__init__(evaluator, similarity, temperature, mode)
        self.item_embeddings: Optional[Sequence[torch.Tensor]] = None    # one table per dataloader (callbacks.py:85-118)
        self._tables: Dict[int, ShardedItemTable] = {}
        self._loss_tables: Dict[int, ShardedItemTable] = {}
        self._log = WeightedMeanLog()
        self.eval_labels = defaultdict(list)
        self.eval_user_embeddings = defaultdict(list)

    def set_item_embeddings(self, item_embeddings: Sequence[torch.Tensor]) -> None:
        self.item_embeddings = item_embeddings
        self._tables = {}
        self._loss_tables = {}

    def on_epoch_start(self) -> None:
        """module.py:421-423, :459-462."""
        self._log = WeightedMeanLog()
        self.eval_labels = defaultdict(list)
        self.eval_user_embeddings = defaultdict(list)

    def step(self, user_encoding: torch.Tensor, labels: torch.Tensor, dataloader_idx: int = 0, stage: str = "val") -> torch.Tensor:
        """One batch of dataloader ``dataloader_idx`` (module.py:425-445, :464-483): score it against that dataloader's
        catalog, evaluate it on its own, log metrics and loss weighted by the batch size.  Returns the batch loss."""
        if self.item_embeddings is None:
            raise RuntimeError("item_embeddings have not been injected")
        if dataloader_idx not in self._tables:
            items = self.item_embeddings[dataloader_idx]
            self._tables[dataloader_idx] = self._table(items)
            self._loss_tables[dataloader_idx] = self._loss_table(items, self._tables[dataloader_idx])
        table = self._tables[dataloader_idx]
        users = self._maybe_normalize(user_encoding.detach()).to(torch.float32)
        self.eval_labels[dataloader_idx].append(labels.detach())
        self.eval_user_embeddings[dataloader_idx].append(users)
        n = int(labels.shape[0])
        queries = self._queries(users, table)
        metrics = self.evaluator.evaluate_embeddings(queries, table, labels, metric_prefix=f"{stage}/", mode=self.mode)
        loss = catalog_cross_entropy(queries, self._loss_tables[dataloader_idx], labels, self.temperature)
        suffix = f"/dataloader_idx_{dataloader_idx}"      # what Lightning appends with several dataloaders
        self._log.log_dict({k + suffix: v for k, v in metrics.items()}, batch_size=n)
        self._log.log(f"{stage}/loss{suffix}", loss, batch_size=n)
        return loss

    def logged_metrics(self) -> Dict[str, torch.Tensor]:
        """``trainer.logged_metrics`` at epoch end: batch-size-weighted means per key."""
        return self._log.compute()

    def on_epoch_end(self, stage: str = "val") -> Dict[str, torch.Tensor]:
        """module.py:447-457 / :493-503: keys ``{stage}/{metric}/dataloader_idx_{i}`` -> ``{stage}/{metric}`` by an
        unweighted mean over the dataloaders (``torch.stack(v).mean()``)."""
        all_metric = defaultdict(list)
        for k, v in self.logged_metrics().items():
            if not k.startswith(f"{stage}/") or k.count("/") != 2:
                continue
            _, metric_name, _ = k.split("/")
            all_metric[metric_name].append(v)
        return {f"{stage}/{k}": torch.stack(v).mean() for k, v in all_metric.items()}
