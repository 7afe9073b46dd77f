"""Cost of the catalog cross-entropy's gradient with respect to the queries on one GPU, N = 1,000,000 items, E = 768,
T = 0.05: at BASELINE config 5 (Q = 65,536) and at a training-sized Q = 4,096.

    python tools/lse_grad_bench.py [--iters 5] [--warmup 1] [--chunks 1024,2048,4096,8192] [--profile OUT.txt]

Cases, timed alternately in one process with CUDA events around each whole call (one round = one call of each case):
    fwd_Q             `catalog_cross_entropy` without a graph (3xTF32)
    fwdbwd_Q_cC       the same loss on queries that require grad, then `backward()`; the backward walks the catalog in
                      chunks of C items (`MR_LSE_GRAD_CHUNK`, the measurement override of the built-in chunk)
    torch_4096        torch's autograd on fp32 logits: rows of 512 queries against the whole catalog, `cross_entropy`
                      and `backward()` per row block (a (4,096, N) logits matrix alone would be 16 GB)
The 6 GB item table does not fit the 126 MB L2, so every call streams it from HBM.  Prints one JSON line with the card's
name and power limit, read in the same run, the median / min / max of each case and the largest row error of the fused
gradient against a chunked fp64 reference at Q = 4,096 for each chunk size (relative to the row's largest entry), and
the same figure for the torch gradient.  --profile writes the kernel time table of one backward at Q = 4,096
(torch.profiler, built-in chunk) to OUT.txt."""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from exclude_bench import gpu_info  # noqa: E402
from mergerec_b200 import _lib  # noqa: E402
from mergerec_b200.evaluator import ShardedItemTable  # noqa: E402
from mergerec_b200.module.recommender.module import catalog_cross_entropy  # noqa: E402

N, E, T, ROWS = 1_000_000, 768, 0.05, 512


def torch_loss_backward(users, items, labels):
    """fp32 logits by row blocks, torch's cross-entropy and autograd: the loss and the query gradient."""
    u = users.detach().requires_grad_(True)
    total = 0.0
    for r0 in range(0, u.shape[0], ROWS):
        logits = u[r0:r0 + ROWS] @ items.T
        loss = torch.nn.functional.cross_entropy(logits / T, labels[r0:r0 + ROWS], reduction="sum") / u.shape[0]
        loss.backward()
        total += float(loss.detach())
    return total, u.grad


def fp64_grad(users, items, labels):
    """The gradient of the mean cross-entropy in fp64, chunked over the catalog."""
    U, step, Q = users.double(), 65536, users.shape[0]
    lse = torch.full((Q,), -float("inf"), dtype=torch.float64, device="cuda")
    for n0 in range(0, N, step):
        lse = torch.logaddexp(lse, torch.logsumexp(U @ items[n0:n0 + step].double().T / T, dim=1))
    acc = torch.zeros_like(U)
    for n0 in range(0, N, step):
        I = items[n0:n0 + step].double()
        acc += torch.exp(U @ I.T / T - lse[:, None]) @ I
    return (acc - items[labels].double()) / (T * Q)


def fused_backward(users, table, labels, chunk):
    os.environ["MR_LSE_GRAD_CHUNK"] = str(chunk)
    u = users.detach().requires_grad_(True)
    loss = catalog_cross_entropy(u, table, labels, T)
    loss.backward()
    return float(loss.detach()), u.grad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--chunks", default="1024,2048,4096,8192")
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()
    _lib.require_cuda()
    torch.backends.cuda.matmul.allow_tf32 = False
    chunks = [int(c) for c in args.chunks.split(",")]
    g = torch.Generator(device="cuda").manual_seed(61)
    items = torch.nn.functional.normalize(torch.randn(N, E, generator=g, device="cuda"), dim=-1)
    users = torch.nn.functional.normalize(torch.randn(65536, E, generator=g, device="cuda"), dim=-1)
    labels = torch.randint(0, N, (65536,), generator=g, device="cuda", dtype=torch.int64)
    table = ShardedItemTable(items)
    small_u, small_l = users[:4096].contiguous(), labels[:4096].contiguous()

    cases = {"fwd_4096": lambda: catalog_cross_entropy(small_u, table, small_l, T),
             "fwd_65536": lambda: catalog_cross_entropy(users, table, labels, T),
             "torch_4096": lambda: torch_loss_backward(small_u, items, small_l)}
    for c in chunks:
        cases[f"fwdbwd_4096_c{c}"] = lambda c=c: fused_backward(small_u, table, small_l, c)
        cases[f"fwdbwd_65536_c{c}"] = lambda c=c: fused_backward(users, table, labels, c)

    want = fp64_grad(small_u, items, small_l)

    def err(got):
        return float(((got.double() - want).abs().max(dim=1).values / want.abs().max(dim=1).values).max())

    loss_t, grad_t = torch_loss_backward(small_u, items, small_l)
    res = {"workload": "catalog_cross_entropy_grad", "N": N, "E": E, "T": T, "iters": args.iters, "loss_torch_4096": loss_t,
           "grad_err_torch": err(grad_t)}
    for c in chunks:
        loss_f, grad_f = fused_backward(small_u, table, small_l, c)
        res[f"grad_err_c{c}"] = err(grad_f)
        res[f"loss_fused_4096_c{c}"] = loss_f
    del grad_t, grad_f, want

    times = {c: [] for c in cases}
    for r in range(args.warmup + args.iters):
        for name, fn in cases.items():
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            if r >= args.warmup:
                times[name].append(a.elapsed_time(b))
    res.update(gpu_info())
    for name, t in times.items():
        med = sorted(t)[len(t) // 2]
        res[name] = {"median_ms": round(med, 3), "min_ms": round(min(t), 3), "max_ms": round(max(t), 3)}
    print(json.dumps(res), flush=True)

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        os.environ.pop("MR_LSE_GRAD_CHUNK", None)
        u = small_u.detach().requires_grad_(True)
        loss = catalog_cross_entropy(u, table, small_l, T)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            loss.backward()
            torch.cuda.synchronize()
        os.makedirs(os.path.dirname(os.path.abspath(args.profile)), exist_ok=True)
        with open(args.profile, "w") as f:
            f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=20, max_name_column_width=100))


if __name__ == "__main__":
    main()
