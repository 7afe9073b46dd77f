"""Cost of the bounded label ranks behind `evaluate_embeddings` at BASELINE config 5 (Q = 65,536 queries against
N = 1,000,000 items, E = 768, 3xTF32, ks = {10, 100}) on one GPU.

    python tools/bounded_rank_bench.py [--iters 5] [--warmup 2] [--sweep]

Cases, timed alternately in one process with CUDA events around each whole call, metric floats on the host included:
    list            the list path: `metrics_from_ids(topk_embeddings(k = 100))`
    rank            `label_ranks()` uncapped, then `metrics_from_ranks`
    bounded         `evaluate_embeddings`: `label_ranks(cap = 100)` (probe, compaction, rest), then `metrics_from_ranks`
    bounded_excl50  the same with 50 random ids per query left out
    top1_list / top1_bounded   every label its row's top-1 (every row stays live: the probe is pure overhead)
    r20_list / r20_bounded     about 20 % of the labels in their row's top 100
The first four use the bench's inputs (half of the queries planted next to their label).  Each case reports the median
and min-max over the iterations, and its metrics must equal the list path's.  `--sweep` then times the probe pass for
MR_SCORE_PROBE_DIV in {128, 64, 32} and, at the default probe, the probe and the compacted rest pass for
MR_SCORE_SPLITS in {1, 2, 3, 4, 6, 8} and the plan's own choice.  The 6 GB item table does not fit the 126 MB L2, so
every call streams it from HBM.  Prints one JSON line with the card's name and power limit, read in the same run."""
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
from mergerec_b200.evaluator import evaluator as evm  # noqa: E402

Q, N, E, K, H = 65536, 1_000_000, 768, 100, 50


def planted(items, frac, seed):
    """The bench's query construction (bench_workloads.EvalCatalog._make_inputs) with `frac` of the queries planted."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    users = torch.randn(Q, E, generator=g, device="cuda")
    labels = torch.randint(0, N, (Q,), generator=g, device="cuda")
    sel = torch.rand(Q, generator=g, device="cuda") < frac
    users = torch.where(sel[:, None], items[labels] + 0.5 * users / E ** 0.5, users)
    return torch.nn.functional.normalize(users, dim=-1), labels


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def stats(t):
    t = sorted(t)
    return {"median_ms": round(t[len(t) // 2], 3), "min_ms": round(t[0], 3), "max_ms": round(t[-1], 3)}


def sweep(ev, queries, table, labels, iters):
    """Pass times of the bounded path's two counting launches under other probe sizes and item splits."""
    from mergerec_b200.evaluator.evaluator import label_score, score_rank
    key = label_score(queries.hi, queries.lo, table, labels)
    out = {"probe_div": {}, "splits": {}}
    for div in ("128", "64", "32"):
        os.environ["MR_SCORE_PROBE_DIV"] = div
        n1 = evm._probe_rows(N)
        out["probe_div"][div] = {"rows": n1, **stats([event_ms(lambda: score_rank(
            queries.hi, queries.lo, table, labels, key, rows=(0, n1))) for _ in range(iters + 1)][1:])}
    os.environ.pop("MR_SCORE_PROBE_DIV")
    n1 = evm._probe_rows(N)
    probe = score_rank(queries.hi, queries.lo, table, labels, key, rows=(0, n1))
    live = torch.nonzero((key != 0) & (probe < K)).flatten()
    hi, lo, lab, k2 = (t[live].contiguous() for t in (queries.hi, queries.lo, labels, key))
    out["live_rows"] = int(live.numel())
    for s in ("0", "1", "2", "3", "4", "6", "8"):
        os.environ["MR_SCORE_SPLITS"] = s
        out["splits"]["plan" if s == "0" else s] = {
            "probe": stats([event_ms(lambda: score_rank(queries.hi, queries.lo, table, labels, key, rows=(0, n1)))
                            for _ in range(iters + 1)][1:]),
            "rest_compacted": stats([event_ms(lambda: score_rank(hi, lo, table, lab, k2, rows=(n1, N)))
                                     for _ in range(iters + 1)][1:])}
    os.environ.pop("MR_SCORE_SPLITS")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sweep", action="store_true")
    args = ap.parse_args()
    _lib.require_cuda()
    g = torch.Generator(device="cuda").manual_seed(99)
    items = torch.nn.functional.normalize(torch.randn(N, E, generator=g, device="cuda"), dim=-1)
    ev = Evaluator(["RECALL", "NDCG"], [10, K])
    table = ShardedItemTable(items)
    users, labels = planted(items, 0.5, 1)
    u20, l20 = planted(items, 0.2, 2)
    l1 = torch.randint(0, N, (Q,), generator=g, device="cuda")
    q, q20, q1 = ev.prepare_queries(users), ev.prepare_queries(u20), ev.prepare_queries(items[l1])
    del users, u20, items
    excl = torch.randint(0, N, (Q, H), generator=g, device="cuda", dtype=torch.int64)

    def lst(qq, ll, exclude=None):
        return lambda: ev.metrics_from_ids(ev.topk_embeddings(qq, table, K, exclude=exclude)[1], ll)

    def bnd(qq, ll, exclude=None):
        return lambda: ev.evaluate_embeddings(qq, table, ll, exclude=exclude)

    cases = {
        "list": lst(q, labels),
        "rank": lambda: ev.metrics_from_ranks(ev.label_ranks(q, table, labels)),
        "bounded": bnd(q, labels),
        "list_excl50": lst(q, labels, excl),
        "bounded_excl50": bnd(q, labels, excl),
        "top1_list": lst(q1, l1),
        "top1_bounded": bnd(q1, l1),
        "r20_list": lst(q20, l20),
        "r20_bounded": bnd(q20, l20),
    }
    results = {name: fn() for name, fn in cases.items()}
    agree = {name: results[name] == results[ref] for name, ref in (
        ("rank", "list"), ("bounded", "list"), ("bounded_excl50", "list_excl50"), ("top1_bounded", "top1_list"),
        ("r20_bounded", "r20_list"))}
    times = {c: [] for c in cases}
    for r in range(args.warmup + args.iters):
        for name, fn in cases.items():
            t = event_ms(fn)
            if r >= args.warmup:
                times[name].append(t)
    res = {"workload": "bounded_rank_cfg5", "Q": Q, "N": N, "E": E, "K": K, "H": H, "iters": args.iters,
           "probe_rows": evm._probe_rows(N), "metrics_agree": agree,
           "metrics": {k: results[k] for k in ("bounded", "top1_bounded", "r20_bounded")}, **gpu_info()}
    for name, t in times.items():
        res[name] = stats(t)
    for name, ref in (("bounded", "list"), ("bounded_excl50", "list_excl50"), ("top1_bounded", "top1_list"),
                      ("r20_bounded", "r20_list"), ("rank", "list")):
        res[name]["vs_list"] = round(res[name]["median_ms"] / res[ref]["median_ms"], 4)
    if args.sweep:
        res["sweep"] = sweep(ev, q, table, labels, args.iters)
    print(json.dumps(res), flush=True)
    if not all(agree.values()):
        sys.exit(f"metrics differ: {agree}")


if __name__ == "__main__":
    main()
