"""Item-table handles for the fused scoring path: the pre-split (hi, lo) TF32 operands of one GPU's shard of the
catalog, and the exchange step that merges per-GPU top-K lists (NCCL allgather over NVLink + `mr_topk_merge`).

The reference is single-GPU and evaluates one domain catalog at a time (README.md:51-53, utils.py:108-119); the
sharding is this package's multi-GPU extension (SURVEY.md section 8(e)): rows [lo, hi) of the item table live on
rank r, global item id = id_base + local row, queries are replicated, and the merged answer is bit-identical to
the single-GPU one because every (query, item) score is computed by the same instruction sequence on any rank.
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import torch

from .. import _lib

MR_SCORE_TF32X3, MR_SCORE_TF32X1, MR_SCORE_BF16 = 0, 1, 2
MAX_FUSED_TOPK = 128


def shard_bounds(n_items: int, world: int, rank: int) -> Tuple[int, int]:
    """Rows [lo, hi) of the item table owned by `rank`: contiguous, sizes differ by at most one, earlier ranks
    take the remainder (so global ids stay ascending with the rank -- the tie rule needs nothing else)."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    base, rem = divmod(n_items, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def split_tf32(x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """hi = rna_tf32(x), lo = rna_tf32(x - hi) on the GPU (`mr_split_tf32`)."""
    dev = _lib.require_cuda()
    lib = _lib.load()
    x = x.to(device=dev, dtype=torch.float32).contiguous()
    hi, lo = torch.empty_like(x), torch.empty_like(x)
    if x.numel():
        _lib.check(lib.mr_split_tf32(_lib.dptr(x), x.numel(), _lib.dptr(hi), _lib.dptr(lo), _lib.stream_handle()),
                   "mr_split_tf32")
    return hi, lo


def to_bf16(x: torch.Tensor) -> torch.Tensor:
    """bf16 copy of an fp32 tensor, round to nearest even (`mr_to_bf16`): the operand of the bf16-compat mode."""
    dev = _lib.require_cuda()
    lib = _lib.load()
    x = x.to(device=dev, dtype=torch.float32).contiguous()
    out = torch.empty(x.shape, dtype=torch.bfloat16, device=dev)
    if x.numel():
        _lib.check(lib.mr_to_bf16(_lib.dptr(x), x.numel(), _lib.dptr(out), _lib.stream_handle()), "mr_to_bf16")
    return out


def replicate_from_host(host: torch.Tensor, group=None) -> torch.Tensor:
    """A host tensor every rank holds (the query embeddings, the labels) -> the same tensor on every rank's GPU, moving
    each byte over PCIe ONCE per node instead of once per rank: rank r uploads rows [r * m, (r + 1) * m) and one NCCL
    all-gather over NVLink (hundreds of GB/s against the ~25 GB/s per rank that eight simultaneous host copies get)
    completes it.  Without a group (or with one rank) it is a plain asynchronous copy."""
    dev = _lib.require_cuda()
    world = 1
    if group is not None:
        import torch.distributed as dist
        world = dist.get_world_size(group)
    if world == 1:
        return host.to(dev, non_blocking=True)
    import torch.distributed as dist
    rank = dist.get_rank(group)
    n = host.shape[0]
    m = (n + world - 1) // world
    full = torch.empty((world * m,) + tuple(host.shape[1:]), dtype=host.dtype, device=dev)
    lo, hi = min(n, rank * m), min(n, (rank + 1) * m)
    mine = full[rank * m:(rank + 1) * m]
    if hi > lo:
        mine[:hi - lo].copy_(host[lo:hi], non_blocking=True)
    # (the send buffer must not alias the receive buffer: one small device copy of this rank's slice)
    dist.all_gather_into_tensor(full, mine.clone(), group=group)
    return full[:n]


def topk_merge(vals: torch.Tensor, ids: torch.Tensor, k_out: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Merge (L, Q, K_in) per-shard lists into (Q, k_out) under (score desc, id asc) (`mr_topk_merge`)."""
    dev = _lib.require_cuda()
    lib = _lib.load()
    vals = vals.to(device=dev, dtype=torch.float32).contiguous()
    ids = ids.to(device=dev, dtype=torch.int32).contiguous()
    L, Q, K_in = vals.shape
    out_v = torch.empty((Q, k_out), dtype=torch.float32, device=dev)
    out_i = torch.empty((Q, k_out), dtype=torch.int32, device=dev)
    _lib.check(lib.mr_topk_merge(_lib.dptr(vals), _lib.dptr(ids), L, Q, K_in, k_out, _lib.dptr(out_v), _lib.dptr(out_i),
                                 _lib.stream_handle()), "mr_topk_merge")
    return out_v, out_i


class ShardedItemTable:
    """One rank's rows of the item-embedding table, stored as the (hi, lo) operand pair of the 3xTF32 contraction.

    items      (n_local, E) fp32 rows owned by this rank (any device; moved to the current GPU).
    id_base    global id of local row 0.
    n_total    catalog size over all ranks (defaults to n_local: a single-GPU table).
    group      torch.distributed process group holding the other shards (None = no exchange).

    The handle also keeps the scratch the scoring kernel needs (`workspace`: candidate buffers and per-split lists,
    sized by `mr_score_topk_workspace_bytes`) and the all-gather landing buffer, so repeated evaluations against the
    same table allocate nothing.
    """

    def __init__(self, items: torch.Tensor, id_base: int = 0, n_total: Optional[int] = None, group=None,
                 normalize: bool = False, bf16: bool = False):
        dev = _lib.require_cuda()
        items = items.to(device=dev, dtype=torch.float32)
        if items.dim() != 2:
            raise ValueError("item table must be (N, E)")
        if normalize:
            items = torch.nn.functional.normalize(items, p=2, dim=-1)  # module/recommender/module.py:74-77
        self.bf16 = bool(bf16)
        if self.bf16:      # bf16-compat mode (the reference's default bf16-mixed runs): one bf16 table, no split
            self.hi, self.lo = to_bf16(items), None
        else:
            self.hi, self.lo = split_tf32(items)
        self.n_local, self.dim = items.shape
        self.id_base = int(id_base)
        self.n_total = int(n_total if n_total is not None else self.n_local)
        self.group = group
        self._ws: Optional[torch.Tensor] = None
        self._gathered: Optional[torch.Tensor] = None

    def workspace(self, nbytes: int) -> torch.Tensor:
        """Scratch of at least `nbytes` on the table's device, kept between calls (grown when needed)."""
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=self.hi.device)
        return self._ws

    def gather_buffer(self, Q: int, k: int) -> torch.Tensor:
        shape = (self.world, 2, Q, k)
        if self._gathered is None or tuple(self._gathered.shape) != shape:
            self._gathered = torch.empty(shape, dtype=torch.int32, device=self.hi.device)
        return self._gathered

    @classmethod
    def from_full(cls, items: torch.Tensor, group=None, normalize: bool = False, bf16: bool = False) -> "ShardedItemTable":
        """Keep this rank's slice of a table every rank can see (host tensor or replicated)."""
        import torch.distributed as dist
        world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
        rank = dist.get_rank(group) if world > 1 else 0
        lo, hi = shard_bounds(items.shape[0], world, rank)
        return cls(items[lo:hi], id_base=lo, n_total=items.shape[0], group=group if world > 1 else None,
                   normalize=normalize, bf16=bf16)

    @property
    def world(self) -> int:
        if self.group is None:
            return 1
        import torch.distributed as dist
        return dist.get_world_size(self.group)

    @property
    def sharded(self) -> bool:
        """The catalog is split over more than one rank: results need a collective over `group`."""
        return self.group is not None and self.world > 1


def topk_merge_packed(packed: torch.Tensor, k_out: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Merge the exchange buffer (L, 2, Q, K_in) int32 -- plane 0 the fp32 score bits, plane 1 the global ids of
    rank l's list -- into (Q, k_out) (`mr_topk_merge_packed`)."""
    dev = _lib.require_cuda()
    lib = _lib.load()
    if packed.dtype != torch.int32 or packed.dim() != 4 or packed.shape[1] != 2 or not packed.is_contiguous():
        raise ValueError("expected a contiguous (L, 2, Q, K) int32 exchange buffer")
    L, _, Q, K_in = packed.shape
    out_v = torch.empty((Q, k_out), dtype=torch.float32, device=dev)
    out_i = torch.empty((Q, k_out), dtype=torch.int32, device=dev)
    _lib.check(lib.mr_topk_merge_packed(_lib.dptr(packed), L, Q, K_in, k_out, _lib.dptr(out_v), _lib.dptr(out_i),
                                        _lib.stream_handle()), "mr_topk_merge_packed")
    return out_v, out_i


def new_packed_list(Q: int, k: int, device) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """One (2, Q, k) int32 buffer and its two planes viewed as the (values fp32, ids int32) outputs of the scoring
    kernel: the kernel writes its result straight into the buffer the all-gather sends."""
    buf = torch.empty((2, Q, k), dtype=torch.int32, device=device)
    return buf, buf[0].view(torch.float32), buf[1]


def exchange_packed(local: torch.Tensor, k: int, group, merge: Optional[Callable] = None,
                    gathered: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """The exchange step: ONE all-gather (NCCL over NVLink) of every rank's (2, Q, k) list buffer, then the merge.
    `merge(vals (L, Q, k), ids (L, Q, k), k)` is injectable so the host logic can run with the gloo backend on CPU
    tensors (tests); the product path (merge=None) uses `mr_topk_merge_packed` on the gathered buffer as it is."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    _, Q, kk = local.shape
    if gathered is None or gathered.shape != (world, 2, Q, kk) or gathered.device != local.device:
        gathered = torch.empty((world, 2, Q, kk), dtype=torch.int32, device=local.device)
    # concatenated form (world * 2 * Q, k): accepted by both the nccl and the gloo backends
    dist.all_gather_into_tensor(gathered.view(world * 2 * Q, kk), local.view(2 * Q, kk), group=group)
    if merge is None:
        return topk_merge_packed(gathered, k)
    return merge(gathered[:, 0].contiguous().view(torch.float32), gathered[:, 1].contiguous(), k)


def exchange_topk(local_vals: torch.Tensor, local_ids: torch.Tensor, k: int, group,
                  merge: Optional[Callable] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """`exchange_packed` for lists held as two separate (Q, k) tensors (packs them with one copy)."""
    import torch.distributed as dist
    if dist.get_world_size(group) == 1:
        return local_vals, local_ids
    local = torch.stack([local_vals.contiguous().view(torch.int32), local_ids.contiguous().to(torch.int32)])
    return exchange_packed(local, k, group, merge)
