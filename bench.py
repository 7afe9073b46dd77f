#!/usr/bin/env python
"""bench.py -- throughput of the MergeRec hot paths on B200, one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input (random-init weights of the named
architecture; there is no network for checkpoints).  `value` is the whole-job throughput with inputs already
in HBM; `e2e` is the same metric through the public API with HOST buffers (pinned) and the host<->device
copies inside the timed region.  `roofline` times the dominant kernel alone with CUDA events;
`cpu_baseline` times the UNMODIFIED reference packages (baseline/_ref, copied there by baseline/install_ref.py) on the
box's host cores, with the oracle port (oracle/) beside it; where baseline/_ref is absent only the port runs and the
line says `kind: "port"`.  `--impl reference` runs only that CPU arm.  See DESIGN.md section "Measurement".
`--dump-outputs DIR` saves what the last timed step returned (the companion's too) as DIR/<name>.npy, larger outputs
as a fixed seeded sample, so that two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


# ------------------------------------------------------------------------------------------------ utilities
_JSON_FD = None


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory: str, outputs: dict) -> None:
    """Write every output as `directory/<name>.npy` (float32 or float64), at most DUMP_LIMIT_BYTES in all: the inputs
    are seeded, so two builds run with the same arguments can be compared array by array."""
    arrays = {name: np.asarray(a) for name, a in outputs.items()}
    for name, a in arrays.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"output {name} is {a.dtype}, not float32 / float64")
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"outputs hold {total} bytes, more than the {DUMP_LIMIT_BYTES} a dump may take")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)
    log(f"wrote {len(arrays)} outputs ({total} bytes) to {directory}")


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=float(p["hbm_gbs"]), bf16_tflops=float(p["bf16_tflops"]),
                    bf16_tflops_sustained=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        threading.Thread(target=self._pump, daemon=True).start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))


def use_all_host_threads() -> int:
    """The CPU arms use every host core: torchrun exports OMP_NUM_THREADS=1 to its workers, which would otherwise
    serialise the OpenMP oracle and numpy's BLAS.  Returns the thread count in effect."""
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        pass
    os.environ["OMP_NUM_THREADS"] = str(n)
    from oracle import oracle as orc
    orc.set_threads(n)
    try:
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=n)
    except Exception:  # noqa: BLE001
        pass
    torch.set_num_threads(n)
    return n


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def event_time_ms(fn, iters: int) -> float:
    """Average device time of fn() over `iters` calls (after one untimed call), CUDA events on the current stream."""
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


# ------------------------------------------------------------------------------------------------ workloads
from bench_workloads import WORKLOADS, DEFAULT_WORKLOAD  # noqa: E402


def measure_tf32_peak(device) -> dict:
    """cuBLAS TF32 GEMM (torch.matmul on fp32 operands with allow_tf32) at 8192^3: best of 10 (burst) and back to back
    for ~2 s (sustained, under the power cap) -- the tensor-pipe denominators of the evaluator's roofline, measured in
    this run on this GPU instead of derived from the bf16 figure."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=device)
        b = torch.randn(n, n, device=device)
        c = torch.empty(n, n, device=device)
        flops = 2.0 * n ** 3
        for _ in range(3):
            torch.matmul(a, b, out=c)
        torch.cuda.synchronize()
        best = 1e30
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(10):
            e0.record()
            torch.matmul(a, b, out=c)
            e1.record()
            e1.synchronize()
            best = min(best, e0.elapsed_time(e1))
        reps = max(10, int(2000.0 / best))
        e0.record()
        for _ in range(reps):
            torch.matmul(a, b, out=c)
        e1.record()
        e1.synchronize()
        sustained = e0.elapsed_time(e1) / reps
        return {"tf32_tflops": flops / (best * 1e-3) / 1e12, "tf32_tflops_sustained": flops / (sustained * 1e-3) / 1e12,
                "how": f"torch.matmul fp32 with allow_tf32 (cuBLAS TF32), {n}^3: best of 10 / {reps} back to back"}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


_L2_FLUSH = None


def flush_l2(device):
    """Write a 512 MB buffer (4x the 126 MB L2) so the next step starts from a cold cache."""
    global _L2_FLUSH
    if _L2_FLUSH is None or _L2_FLUSH.device != device:
        _L2_FLUSH = torch.empty(512 << 20, dtype=torch.uint8, device=device)
    _L2_FLUSH.fill_(1)


def measure(wl, steps: int, warmup: int, rank: int, world: int, local_rank: int, cpu_arm: bool, sample_clocks: bool,
            outputs: dict = None):
    """One workload through the bench contract: W untimed warm-up steps, exactly K timed steps between barrier +
    synchronize pairs (CUDA events, max over ranks), the end-to-end arm (pinned host inputs, host<->device copies in
    the timed region), the roofline of the dominant kernel and the CPU arm.  Returns the JSON line (rank 0) or None.
    `outputs`, when given, receives the host arrays that the last timed step computed (`wl.outputs()`)."""
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    wl.setup()
    # clocks are sampled from the first warm-up step to the end of the last measured loop (the timed region
    # itself can be a few ms, shorter than one nvidia-smi sample period)
    sampler = ClockSampler(local_rank) if (sample_clocks and rank == 0) else None
    if sampler:
        sampler.start()
    for _ in range(warmup):
        wl.step()
    barrier()
    if getattr(wl, "l2_flush", False):
        # inputs that fit L2: flush between the timed steps and time every step with its own event pair
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in evs:
            flush_l2(wl.device)
            a.record()
            wl.step()
            b.record()
        barrier()
        total_ms = reduce_max(sum(a.elapsed_time(b) for a, b in evs))
    else:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            wl.step()
        ev1.record()
        barrier()
        total_ms = reduce_max(ev0.elapsed_time(ev1))
    if hasattr(wl, "finish"):
        wl.finish()   # deferred host-side checks of the timed steps, checksums, stage timings (every rank)
    if outputs is not None:
        outputs.update(wl.outputs())     # before the end-to-end arm overwrites the step's buffers

    # end to end through the public API: pinned host inputs -> H2D -> kernels -> D2H result, every step
    wl.setup_e2e()
    for _ in range(min(warmup, 2)):
        wl.step_e2e()
    barrier()
    e2e_steps = max(1, min(steps, wl.e2e_steps_cap))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    for _ in range(e2e_steps):
        wl.step_e2e()
    ev1.record()
    barrier()
    e2e_wall = time.perf_counter() - t0
    e2e_ms = reduce_max(max(ev0.elapsed_time(ev1), e2e_wall * 1e3)) / e2e_steps
    if hasattr(wl, "teardown_e2e"):
        wl.teardown_e2e()

    roof = wl.roofline(measured_peaks()) if rank == 0 else None
    clocks = sampler.stop() if sampler else None
    cpu = None
    if rank == 0 and cpu_arm:
        use_all_host_threads()
        cpu = wl.cpu_baseline()
    if rank != 0:
        return None
    ms_per_step = total_ms / steps
    units = wl.units_per_step_all_ranks()
    line = {
        "metric": wl.metric, "value": units / (ms_per_step * 1e-3), "unit": wl.unit, "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": wl.scaling, "vs_baseline": None, "dtype": wl.dtype, "data": "synthetic",
        "config": wl.config(),
        "e2e": {"value": units / (e2e_ms * 1e-3), "unit": wl.unit, "h2d_bytes_per_step": wl.h2d_bytes,
                "d2h_bytes_per_step": wl.d2h_bytes, "ms_per_step": e2e_ms, "steps": e2e_steps},
        "gpu_launches": wl.launches_per_step * steps,
        "roofline": roof,
    }
    if clocks is not None:
        line["clocks"] = clocks
    if cpu is not None:
        line["cpu_baseline"] = cpu
    line.update(wl.extra())
    if hasattr(wl, "Q"):
        line["eval_seqs_per_s"] = wl.Q / (ms_per_step * 1e-3)
    return line


def run_ours(args):
    rank, local_rank, world = dist_env()
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run for --gpus > 1")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    cpu_arm = world == 1 and not args.no_cpu_baseline
    outputs = {} if (args.dump_outputs and rank == 0) else None
    wl = WORKLOADS[args.workload](rank=rank, world=world, device=device)
    line = measure(wl, args.steps, args.warmup, rank, world, local_rank, cpu_arm, sample_clocks=True, outputs=outputs)
    # the other hot path, carried beside the headline: the merger at the size BASELINE.json quotes it on (single GPU)
    # or its sharded form (several GPUs) -- a complete nested line with its own roofline / e2e / cpu_baseline
    comp_cls = None if args.no_companion else wl.companion()
    if comp_cls is not None:
        wl.release()
        del wl
        torch.cuda.empty_cache()
        comp = comp_cls(rank=rank, world=world, device=device)
        comp_outputs = None if outputs is None else {}
        try:
            sub = measure(comp, min(args.steps, 20), max(3, min(args.warmup, 5)), rank, world, local_rank, cpu_arm,
                          sample_clocks=False, outputs=comp_outputs)
        except Exception as e:  # noqa: BLE001 -- the headline line must still be printed
            if world > 1:
                raise
            sub = {"error": repr(e)}
        if rank == 0:
            line[comp.companion_key] = sub
        if comp_outputs:
            outputs.update({f"{comp.companion_key}.{name}": a for name, a in comp_outputs.items()})
    if rank == 0:
        emit(line)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.destroy_process_group()


def run_reference(args):
    """The reference's own CPU implementation of the path on the box's host cores, all host threads, same metric /
    config: the UNMODIFIED reference packages from baseline/_ref when they are installed (`kind: "reference"`), else the
    oracle port (`kind: "port"`).  Every step is a bounded sample of the workload, actually run W + K times."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    use_all_host_threads()
    wl = WORKLOADS[args.workload](rank=0, world=1, device=None)
    res = wl.reference_arm(steps=args.steps, warmup=args.warmup)
    line = {
        "impl": "reference", "metric": wl.metric, "value": res["value"], "unit": wl.unit, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": wl.scaling, "vs_baseline": None, "dtype": wl.dtype, "data": "synthetic", "config": wl.config(),
        "cpu_baseline": {"value": res["value"], "unit": wl.unit, "cores": res["cores"], "kind": res.get("kind", "port"),
                         "sample": res["sample"]},
        "e2e": {"value": res["value"], "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def main():
    # Only the JSON line may reach stdout: libraries (NCCL with NCCL_DEBUG set, ...) print there from C code, so
    # file descriptor 1 is pointed at stderr for the whole run and the line is written to the saved descriptor.
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-companion", action="store_true", help="skip the nested merger line of the evaluator workloads")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (the companion's as <key>.<name>)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        log("note: fewer than 3 warm-up steps requested; the timing rules ask for >= 3")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
