"""Multi-GPU worker of tests/test_nccl_label_rank_gpu.py: one process per GPU under torch.distributed.run, NCCL backend.

`Evaluator.label_ranks` on a row-sharded item table (two all-reduces of Q words: MAX of the label keys, SUM of the
counts) must give every rank the ranks of the single-GPU call, and large-k metrics must equal the single-GPU ones.
Exit code 0 = all checks passed on every rank."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mergerec_b200 import synth  # noqa: E402
from mergerec_b200.evaluator import MR_SCORE_BF16, MR_SCORE_TF32X3, Evaluator, ShardedItemTable  # noqa: E402


def main() -> int:
    rank, local_rank = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=dev)
    ok = True
    try:
        for kind, Q, N, E in (("grid", 300, 20011, 64), ("gauss", 520, 50021, 768)):
            users, items, labels = synth.make_catalog(Q, N, E, kind=kind, seed=41)
            tu, ti, tl = (torch.from_numpy(a).to(dev) for a in (users, items, labels))
            tl[::7] = -1
            excl = torch.randint(0, N, (Q, 30), device=dev, generator=torch.Generator(device=dev).manual_seed(42))
            excl[::5, 0] = tl[::5]
            ev = Evaluator(["NDCG", "RECALL"], [10, 200, N])
            for mode in (MR_SCORE_TF32X3, MR_SCORE_BF16):
                bf16 = mode == MR_SCORE_BF16
                q = ev.prepare_queries(tu, mode=mode)
                full = ShardedItemTable(ti, bf16=bf16)
                table = ShardedItemTable.from_full(ti, group=dist.group.WORLD, bf16=bf16)
                for exclude in (None, excl):
                    want = ev.label_ranks(q, full, tl, mode=mode, exclude=exclude)
                    got = ev.label_ranks(q, table, tl, mode=mode, exclude=exclude)
                    ok &= bool(torch.equal(got, want))
                    ok &= ev.evaluate_embeddings(q, table, tl, mode=mode, exclude=exclude) == \
                        ev.evaluate_embeddings(q, full, tl, mode=mode, exclude=exclude)
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = bool(flag.item())
    finally:
        dist.destroy_process_group()
    if rank == 0:
        print("nccl label-rank worker: ok" if ok else "nccl label-rank worker: FAILED")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
