"""Cost of leaving items out of the ranking inside the fused scoring kernel, at BASELINE config 5 (Q = 65,536 queries
against N = 1,000,000 items, E = 768, K = 100, 3xTF32) on one GPU.

    python tools/exclude_bench.py [--iters 5] [--warmup 2]

Cases, timed alternately in one process with CUDA events (one round = one call of each case, so drift of the clocks or
of the neighbours' load spreads over all of them):
    none         mr_score_topk, no exclusion
    empty        mr_score_topk_exclude, every row's list empty
    random50     H = 50 uniformly random item ids per query
    adversarial  H = 50: each row's own unfiltered top-50, so every excluded item survives the threshold filter
The 6 GB item table does not fit the 126 MB L2, so every call streams it from HBM.  Prints one JSON line with the card's
name and power limit, read in the same run, and checks that the first 50 entries of the adversarial list are positions
50..99 of the unfiltered top-100."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mergerec_b200 import _lib  # noqa: E402
from mergerec_b200.evaluator import ShardedItemTable  # noqa: E402
from mergerec_b200.evaluator.evaluator import _device_csr, _score_topk  # noqa: E402
from mergerec_b200.evaluator.sharded import MR_SCORE_TF32X3, split_tf32  # noqa: E402

Q, N, E, K, H = 65536, 1_000_000, 768, 100, 50


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"nvidia-smi unavailable: {e}"
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    _lib.require_cuda()
    g = torch.Generator(device="cuda").manual_seed(5)
    users = torch.nn.functional.normalize(torch.randn(Q, E, generator=g, device="cuda"), dim=-1)
    items = torch.nn.functional.normalize(torch.randn(N, E, generator=g, device="cuda"), dim=-1)
    u_hi, u_lo = split_tf32(users)
    del users
    table = ShardedItemTable(items)
    del items
    out = (torch.empty((Q, K), dtype=torch.float32, device="cuda"), torch.empty((Q, K), dtype=torch.int32, device="cuda"))

    dev = u_hi.device
    _, top = _score_topk(u_hi, u_lo, table, K, MR_SCORE_TF32X3, None, None)
    cases = {
        "none": None,
        "empty": _device_csr(torch.full((Q, 1), -1, dtype=torch.int32, device=dev), Q, dev),
        "random50": _device_csr(torch.randint(0, N, (Q, H), generator=g, device=dev), Q, dev),
        "adversarial": _device_csr(top[:, :H], Q, dev),
    }
    _score_topk(u_hi, u_lo, table, K, MR_SCORE_TF32X3, out, cases["adversarial"])
    check = bool(torch.equal(out[1][:, :K - H], top[:, H:]))

    times = {c: [] for c in cases}
    for r in range(args.warmup + args.iters):
        for name, csr in cases.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            _score_topk(u_hi, u_lo, table, K, MR_SCORE_TF32X3, out, csr)
            b.record()
            b.synchronize()
            if r >= args.warmup:
                times[name].append(a.elapsed_time(b))
    res = {"workload": "exclude_cfg5", "Q": Q, "N": N, "E": E, "K": K, "H": H, "iters": args.iters,
           "adversarial_equals_unfiltered_slice": check, **gpu_info()}
    base = sorted(times["none"])[len(times["none"]) // 2]
    for name, t in times.items():
        med = sorted(t)[len(t) // 2]
        res[name] = {"median_ms": round(med, 3), "min_ms": round(min(t), 3), "max_ms": round(max(t), 3),
                     "vs_none": round(med / base, 4)}
    print(json.dumps(res), flush=True)
    if not check:
        sys.exit("the adversarial list does not continue the unfiltered list")


if __name__ == "__main__":
    main()
