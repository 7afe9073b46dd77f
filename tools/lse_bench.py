"""Cost of the catalog cross-entropy at BASELINE config 5 (Q = 65,536 queries against N = 1,000,000 items, E = 768,
T = 0.05) on one GPU.

    python tools/lse_bench.py [--iters 5] [--warmup 2]

Cases, timed alternately in one process with CUDA events around each whole call (one round = one call of each case):
    matrix        the removed loss path, restated: (4,096, N) fp32 logits chunks from `mr_scores_fp32` (CUDA cores)
                  + torch's `cross_entropy`, summed over the chunks
    lse           `label_log_softmax` (3xTF32) and the fp64 mean: the loss path of `catalog_cross_entropy`
    rank          `label_ranks` (3xTF32): the same tensor work with the counting epilogue, as the reference point
    lse_excl50    `label_log_softmax` with 50 random ids per query left out
    lse_bf16      `label_log_softmax` in the bf16-compat mode
The 6 GB item table does not fit the 126 MB L2, so every call streams it from HBM.  Prints one JSON line with the card's
name and power limit, read in the same run, and the loss of the matrix path and of the fused path side by side."""
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
from mergerec_b200.evaluator import MR_SCORE_BF16, Evaluator, ShardedItemTable  # noqa: E402

Q, N, E, H, T, ROWS = 65536, 1_000_000, 768, 50, 0.05, 4096


def matrix_loss(users, items, labels):
    """The loss path this change removed from `catalog_cross_entropy`."""
    lib = _lib.load()
    total = torch.zeros((), dtype=torch.float32, device="cuda")
    logits = torch.empty((ROWS, N), dtype=torch.float32, device="cuda")
    for r0 in range(0, Q, ROWS):
        _lib.check(lib.mr_scores_fp32(_lib.dptr(users[r0:r0 + ROWS]), ROWS, _lib.dptr(items), N, E, _lib.dptr(logits), N,
                                      _lib.stream_handle()), "mr_scores_fp32")
        total = total + torch.nn.functional.cross_entropy(logits / T, labels[r0:r0 + ROWS], reduction="sum")
    return total / Q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    _lib.require_cuda()
    g = torch.Generator(device="cuda").manual_seed(52)
    users = torch.nn.functional.normalize(torch.randn(Q, E, generator=g, device="cuda"), dim=-1)
    items = torch.nn.functional.normalize(torch.randn(N, E, generator=g, device="cuda"), dim=-1)
    labels = torch.randint(0, N, (Q,), generator=g, device="cuda", dtype=torch.int64)
    ev = Evaluator(["RECALL"], [10])
    queries, table = ev.prepare_queries(users), ShardedItemTable(items)
    queries16, table16 = ev.prepare_queries(users, mode=MR_SCORE_BF16), ShardedItemTable(items, bf16=True)
    _, top = ev.topk_embeddings(queries, table, 100)
    labels[::2] = top[::2, 7].to(torch.int64)           # half of the labels among each query's best 100
    excl = torch.randint(0, N, (Q, H), generator=g, device="cuda", dtype=torch.int64)
    del top

    def fused_loss(q, t, mode=0, exclude=None):
        return -ev.label_log_softmax(q, t, labels, T, mode=mode, exclude=exclude).to(torch.float64).mean()

    cases = {
        "matrix": lambda: matrix_loss(users, items, labels),
        "lse": lambda: fused_loss(queries, table),
        "rank": lambda: ev.label_ranks(queries, table, labels),
        "lse_excl50": lambda: fused_loss(queries, table, exclude=excl),
        "lse_bf16": lambda: fused_loss(queries16, table16, MR_SCORE_BF16),
    }
    loss_matrix, loss_lse = float(cases["matrix"]()), float(cases["lse"]())
    loss_bf16 = float(cases["lse_bf16"]())

    times = {c: [] for c in cases}
    for r in range(args.warmup + args.iters):
        for name, fn in cases.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            if r >= args.warmup:
                times[name].append(a.elapsed_time(b))
    res = {"workload": "catalog_cross_entropy_cfg5", "Q": Q, "N": N, "E": E, "H": H, "T": T, "iters": args.iters,
           "loss_matrix": loss_matrix, "loss_lse": loss_lse, "loss_lse_bf16": loss_bf16,
           "loss_rel_diff": abs(loss_lse - loss_matrix) / abs(loss_matrix), **gpu_info()}
    base = sorted(times["matrix"])[len(times["matrix"]) // 2]
    for name, t in times.items():
        med = sorted(t)[len(t) // 2]
        res[name] = {"median_ms": round(med, 3), "min_ms": round(min(t), 3), "max_ms": round(max(t), 3),
                     "vs_matrix": round(med / base, 4)}
    print(json.dumps(res), flush=True)
    if not res["loss_rel_diff"] <= 1e-5:
        sys.exit(f"losses differ: matrix {loss_matrix} fused {loss_lse}")


if __name__ == "__main__":
    main()
