"""Multi-GPU worker of tests/test_nccl_label_log_softmax_gpu.py: one process per GPU under torch.distributed.run, NCCL
backend.

`Evaluator.label_log_softmax` on a row-sharded item table (an all-reduce MAX of the label keys, one all-gather of the
(shift, sum) partials, merged in rank order) must give every rank the same bits, equal to the single-GPU call within
1e-6 * max(1, |x|).  Exit code 0 = all checks passed on every rank."""
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
    world = dist.get_world_size()
    ok = True
    try:
        for kind, Q, N, E in (("grid", 300, 20011, 64), ("gauss", 520, 50021, 768)):
            users, items, labels = synth.make_catalog(Q, N, E, kind=kind, seed=43)
            tu, ti, tl = (torch.from_numpy(a).to(dev) for a in (users, items, labels))
            tl[::7] = -1
            excl = torch.randint(0, N, (Q, 30), device=dev, generator=torch.Generator(device=dev).manual_seed(44))
            excl[::5, 0] = tl[::5]
            for mode in (MR_SCORE_TF32X3, MR_SCORE_BF16):
                bf16 = mode == MR_SCORE_BF16
                q = Evaluator.prepare_queries(tu, mode=mode)
                full = ShardedItemTable(ti, bf16=bf16)
                table = ShardedItemTable.from_full(ti, group=dist.group.WORLD, bf16=bf16)
                for exclude in (None, excl):
                    want = Evaluator.label_log_softmax(q, full, tl, 0.05, mode=mode, exclude=exclude)
                    got = Evaluator.label_log_softmax(q, table, tl, 0.05, mode=mode, exclude=exclude)
                    same_nan = torch.equal(got.isnan(), want.isnan())
                    fin = want.isfinite()
                    err = ((got - want).abs()[fin].double() / want[fin].abs().double().clamp(min=1.0)).max()
                    ok &= bool(same_nan and torch.equal(got[want.isinf()], want[want.isinf()]) and err <= 1e-6)
                    every = [torch.empty_like(got) for _ in range(world)]
                    dist.all_gather(every, got)
                    ok &= all(torch.equal(e.view(torch.int32), got.view(torch.int32)) for e in every)
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = bool(flag.item())
    finally:
        dist.destroy_process_group()
    if rank == 0:
        print("nccl label-log-softmax worker: ok" if ok else "nccl label-log-softmax worker: FAILED")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
