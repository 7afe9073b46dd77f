"""Multi-GPU worker of tests/test_sharded_pcb_gpu.py::test_sharded_pcb_and_dare_over_nccl: one process per GPU under
torch.distributed.run, NCCL backend.  The sharded PCB vectors / merge and the sharded DARE merge must equal, on every
rank's columns, the single-GPU functions run by every rank on the whole vector; the merged bits' integer checksum,
summed over the ranks, must equal rank 0's single-GPU checksum; `ShardedModelMerger.merge("pcb" | "dare")` must return
the `ModelMerger` state_dict on every rank.  Exit code 0 = all checks passed on every rank."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mergerec_b200 import synth  # noqa: E402
from mergerec_b200.merger import ModelMerger  # noqa: E402
from mergerec_b200.merger.algorithms.dare import merge_dare  # noqa: E402
from mergerec_b200.merger.algorithms.pcb import get_pcb_vectors, merge_pcb  # noqa: E402
from mergerec_b200.merger.sharded import (ShardedModelMerger, flat_shard_bounds, get_pcb_vectors_sharded,  # noqa: E402
                                          merge_dare_sharded, merge_pcb_sharded)


def _bits(t):
    return t.contiguous().view(torch.int32)


def main() -> int:
    rank, local_rank, world = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=dev)
    group = dist.group.WORLD
    ok = True
    try:
        # flat vectors: the fast search (with a d mod 32 = 2 tail), the dense search, quantised inputs, d < 100
        for d, K, quant in ((1_000_034, 8, 0.0), (50_021, 5, 0.0), (300_007, 6, 2.5e-4), (64, 3, 0.0)):
            base, models = synth.make_flat(d, K, seed=d % 1000, quantize=quant)
            tb, tm = torch.from_numpy(base).to(dev), [torch.from_numpy(m).to(dev) for m in models]
            lo, hi = flat_shard_bounds(d, world, rank)
            bl, ml = tb[lo:hi].clone(), [m[lo:hi].clone() for m in tm]
            full = get_pcb_vectors(tb, tm, density=0.2)
            part = get_pcb_vectors_sharded(bl, ml, 0.2, d, group)
            ok &= bool(torch.equal(_bits(part[:, :hi - lo]), _bits(full[:, lo:hi])))
            w = [0.3 + 0.1 * i for i in range(K)]
            fullm = merge_pcb(tb, tm, w, density=0.2)
            partm = merge_pcb_sharded(bl, ml, w, 0.2, d, group)
            ok &= bool(torch.equal(_bits(partm), _bits(fullm[lo:hi])))
            chk = _bits(partm).to(torch.int64).sum().reshape(1)
            dist.all_reduce(chk, group=group)
            want = torch.tensor([int(_bits(fullm).to(torch.int64).sum())], device=dev)
            dist.broadcast(want, 0, group=group)                   # rank 0's single-GPU checksum
            ok &= int(chk.item()) == int(want.item())
            masks = torch.rand((K, d), generator=torch.Generator(device=dev).manual_seed(7), device=dev) >= 0.1
            ok &= bool(torch.equal(_bits(merge_dare_sharded(bl, ml, w, 0.1, d, masks=masks, group=group)),
                                   _bits(merge_dare(tb, tm, w, 0.1, masks=masks)[lo:hi])))
            a = merge_dare_sharded(bl, ml, w, 0.1, d, generator=torch.Generator(device=dev).manual_seed(3), group=group)
            b = merge_dare(tb, tm, w, 0.1, generator=torch.Generator(device=dev).manual_seed(3))
            ok &= bool(torch.equal(_bits(a), _bits(b[lo:hi])))
        # the merger front door on a tiny Recformer state_dict
        shapes = synth.tiny_shapes(recformer=True)
        base, models = synth.make_state_dicts(shapes, 5, seed=22, sigma=1e-2)
        to_t = lambda sd: {k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}  # noqa: E731
        base, models = to_t(base), [to_t(m) for m in models]
        ref, sh = ModelMerger(models, base), ShardedModelMerger(models, base, group=group)
        masks = torch.rand((5, ref.models[0].numel()), generator=torch.Generator().manual_seed(1)) >= 0.1
        for mt, kw in (("pcb", dict(density=0.2)), ("dare", dict(density=0.1, masks=masks))):
            x, y = ref.merge(mt, 0.3, **kw), sh.merge(mt, 0.3, **kw)
            ok &= list(x.keys()) == list(y.keys()) and all(torch.equal(x[k], y[k]) for k in x)
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = bool(flag.item())
    finally:
        dist.destroy_process_group()
    if rank == 0:
        print("nccl pcb worker:", "ok" if ok else "MISMATCH", f"(world {world})")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
