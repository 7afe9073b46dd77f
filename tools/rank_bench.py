"""Cost of the label rank against the whole catalog, at BASELINE config 5 (Q = 65,536 queries against N = 1,000,000
items, E = 768, 3xTF32) on one GPU.

    python tools/rank_bench.py [--iters 5] [--warmup 2]

Cases, timed alternately in one process with CUDA events around each whole call (one round = one call of each case):
    topk100      today's metric path: `topk_embeddings(k = 100)` (`mr_score_topk` + merge) plus `label_rank`
    rank         `label_ranks`: the label-score pass and the counting pass, no list
    rank_excl50  `label_ranks` with 50 random ids per query left out
The 6 GB item table does not fit the 126 MB L2, so every call streams it from HBM.  Prints one JSON line with the card's
name and power limit, read in the same run, and checks that Recall / NDCG@{10, 100} agree between the two paths."""
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
from mergerec_b200.evaluator import Evaluator, ShardedItemTable  # noqa: E402
from mergerec_b200.evaluator.metrics import label_rank  # noqa: E402

Q, N, E, K, H = 65536, 1_000_000, 768, 100, 50


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    _lib.require_cuda()
    g = torch.Generator(device="cuda").manual_seed(5)
    users = torch.nn.functional.normalize(torch.randn(Q, E, generator=g, device="cuda"), dim=-1)
    items = torch.nn.functional.normalize(torch.randn(N, E, generator=g, device="cuda"), dim=-1)
    labels = torch.randint(0, N, (Q,), generator=g, device="cuda", dtype=torch.int64)
    ev = Evaluator(["RECALL", "NDCG"], [10, 100])
    queries = ev.prepare_queries(users)
    table = ShardedItemTable(items)
    del users, items
    # half of the labels among each query's best 100, so that the metrics are not all zero
    _, top = ev.topk_embeddings(queries, table, K)
    labels[::2] = top[::2, 7].to(torch.int64)
    excl = torch.randint(0, N, (Q, H), generator=g, device="cuda", dtype=torch.int64)

    cases = {
        "topk100": lambda: label_rank(ev.topk_embeddings(queries, table, K)[1], labels),
        "rank": lambda: ev.label_ranks(queries, table, labels),
        "rank_excl50": lambda: ev.label_ranks(queries, table, labels, exclude=excl),
    }
    m_list = ev.metrics_from_ranks(cases["topk100"]())
    m_rank = ev.metrics_from_ranks(cases["rank"]())
    agree = m_list == m_rank

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
    res = {"workload": "label_rank_cfg5", "Q": Q, "N": N, "E": E, "K": K, "H": H, "iters": args.iters,
           "metrics_agree": agree, "metrics": m_rank, **gpu_info()}
    base = sorted(times["topk100"])[len(times["topk100"]) // 2]
    for name, t in times.items():
        med = sorted(t)[len(t) // 2]
        res[name] = {"median_ms": round(med, 3), "min_ms": round(min(t), 3), "max_ms": round(max(t), 3),
                     "vs_topk100": round(med / base, 4)}
    print(json.dumps(res), flush=True)
    if not agree:
        sys.exit(f"metrics differ: list {m_list} ranks {m_rank}")


if __name__ == "__main__":
    main()
