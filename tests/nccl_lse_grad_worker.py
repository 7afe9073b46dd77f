"""Multi-GPU worker of tests/test_nccl_lse_grad_gpu.py: one process per GPU under torch.distributed.run, NCCL backend.

The backward of `Evaluator.label_log_softmax` on a row-sharded item table (each rank's part, one all-gather of the
(G, Q, E) parts, added in rank order) must give every rank the same bits, equal to the parts of the shards computed on
one GPU and added in rank order, and within 2e-5 of the row maximum of the single-table gradient.  Exit code 0 = all
checks passed on every rank."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mergerec_b200.evaluator import MR_SCORE_TF32X3, Evaluator, ShardedItemTable  # noqa: E402
from mergerec_b200.evaluator.evaluator import _device_csr, _ordered_sum, score_lse_grad  # noqa: E402
from mergerec_b200.evaluator.sharded import shard_bounds  # noqa: E402


def main() -> int:
    rank, local_rank = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=dev)
    world = dist.get_world_size()
    ok = True
    try:
        for Q, N, E, T in ((300, 20011, 64, 0.05), (520, 50021, 768, 1.0)):
            gen = torch.Generator(device=dev).manual_seed(43)
            items = torch.randn(N, E, device=dev, generator=gen)
            users = torch.randn(Q, E, device=dev, generator=gen) * (2.0 * T / E ** 0.5)
            labels = torch.randint(0, N, (Q,), device=dev, generator=gen)
            g = torch.randn(Q, device=dev, generator=gen)
            excl = torch.randint(0, N, (Q, 30), device=dev, generator=gen)
            excl[::5, 0] = labels[::5]
            table = ShardedItemTable.from_full(items, group=dist.group.WORLD)
            for exclude in (None, excl):
                u = users.clone().requires_grad_(True)
                Evaluator.label_log_softmax(u, table, labels, T, exclude=exclude).backward(g)
                got = u.grad
                # single GPU: the same backward on the whole table, and the shards' parts added in rank order
                u1 = users.clone().requires_grad_(True)
                logp = Evaluator.label_log_softmax(u1, items, labels, T, exclude=exclude)
                logp.backward(g)
                q = Evaluator.prepare_queries(users)
                _, (lab, csr, (shift, sums)) = Evaluator._label_log_softmax(
                    q, ShardedItemTable(items), labels, T, MR_SCORE_TF32X3, exclude)
                # the sharded forward's partials: one per shard, each over that shard's rows
                from mergerec_b200.evaluator.evaluator import score_lse
                parts = []
                for r in range(world):
                    lo, hi = shard_bounds(N, world, r)
                    parts.append(score_lse(q.hi, q.lo, ShardedItemTable(items[lo:hi], id_base=lo, n_total=N), T,
                                           MR_SCORE_TF32X3, _device_csr(exclude, Q, dev)))
                shift = torch.stack([p[0] for p in parts]).contiguous()
                sums = torch.stack([p[1] for p in parts]).contiguous()
                gg = torch.where(logp.detach().isfinite(), g, torch.zeros_like(g))
                local = []
                for r in range(world):
                    lo, hi = shard_bounds(N, world, r)
                    local.append(score_lse_grad(q.hi, q.lo, ShardedItemTable(items[lo:hi], id_base=lo, n_total=N), T,
                                                lab, shift, sums, gg, _device_csr(exclude, Q, dev)))
                emulated = _ordered_sum(torch.stack(local))
                ok &= torch.equal(got.view(torch.int32), emulated.view(torch.int32))
                want = u1.grad.double()
                err = (got.double() - want).abs().max(dim=1).values
                ok &= bool((err <= 2e-5 * want.abs().max(dim=1).values).all())
                every = [torch.empty_like(got) for _ in range(world)]
                dist.all_gather(every, got)
                ok &= all(torch.equal(e.view(torch.int32), got.view(torch.int32)) for e in every)
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = bool(flag.item())
    finally:
        dist.destroy_process_group()
    if rank == 0:
        print("nccl lse-grad worker: ok" if ok else "nccl lse-grad worker: FAILED")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
