"""Workloads of bench.py: each is one BASELINE.json configuration, built from synthetic inputs of the named
shapes.  Algorithmic byte counts follow SURVEY.md section 8(d) / DESIGN.md "Measurement"."""
from __future__ import annotations

import os
import time
from typing import Dict, Optional

import numpy as np
import torch

from mergerec_b200 import synth

GB = 1e9


class Workload:
    name = ""
    metric = ""
    unit = ""
    dtype = "f32"
    scaling = "weak"
    launches_per_step = 0
    e2e_steps_cap = 5
    h2d_bytes = 0
    d2h_bytes = 0

    def __init__(self, rank: int, world: int, device: Optional[torch.device]):
        self.rank, self.world, self.device = rank, world, device

    companion_key = "merger"

    def extra(self) -> Dict:
        return {}

    def companion(self):
        """Workload class of the OTHER hot path to carry beside this line (nested, complete), or None."""
        return None

    def release(self) -> None:
        """Drop every device tensor (called before a companion workload is set up)."""
        for name in list(vars(self)):
            if name not in ("rank", "world", "device"):
                delattr(self, name)

    def outputs(self) -> Dict[str, np.ndarray]:
        """What the last timed step handed to its caller, as float32 / float64 host arrays by name (`bench.py
        --dump-outputs`)."""
        raise NotImplementedError(f"workload {self.name} does not name its outputs")


def reference_package():
    """The unmodified reference hot-path packages installed under baseline/_ref (baseline/install_ref.py), or None."""
    import importlib.util
    here = os.path.dirname(os.path.abspath(__file__))
    spec = importlib.util.spec_from_file_location("mr_install_ref", os.path.join(here, "baseline", "install_ref.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    try:
        return mod.load()
    except Exception as e:  # noqa: BLE001 -- a broken copy falls back to the port, and says so
        print(f"[bench] baseline/_ref could not be imported ({type(e).__name__}: {e}); using the oracle port", file=__import__("sys").stderr)
        return None


def timed_steps(fn, steps: int, warmup: int):
    """Run fn() warmup + steps times; (mean seconds per timed step, list of step times)."""
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.mean(ts)), ts


def ncu_traffic(kernel: str):
    """(bytes per launch, source file) of the committed ncu --set full capture of `kernel`, or (None, None)."""
    import json
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")) as f:
            e = json.load(f).get(kernel)
        return (e["bytes"], e["source"]) if e else (None, None)
    except (OSError, ValueError, KeyError):
        return None, None


def _with_traffic(roof: Dict, kernel: str) -> Dict:
    roof["traffic"], src = ncu_traffic(kernel)
    if src:
        roof["traffic_source"] = src
    return roof


def _pinned(t: torch.Tensor) -> torch.Tensor:
    out = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    out.copy_(t)
    return out


OUTPUT_SAMPLE = 1 << 21     # elements kept of a larger output (8 MB of float32), so that a dump stays small


def _output(t: torch.Tensor) -> np.ndarray:
    """`t` as a float32 host array.  Above OUTPUT_SAMPLE elements: the flattened tensor at OUTPUT_SAMPLE positions drawn
    with a fixed seed (ascending), the same positions in every run of the same workload."""
    t = t.detach()
    if t.numel() > OUTPUT_SAMPLE:
        pos = np.sort(np.random.Generator(np.random.PCG64(0)).choice(t.numel(), OUTPUT_SAMPLE, replace=False))
        t = t.reshape(-1)[torch.from_numpy(pos).to(t.device)]
    return t.float().cpu().numpy()


class LambdaMergeK8(Workload):
    """Per-layer lambda merge of 8 BLaIR-base task vectors (the merge half of BASELINE config 2; A4).
    Algorithmic bytes per step: (K+2) * d * 4 (read base + K task-vector rows, write merged)."""

    name = "lambda_merge_k8"
    metric = "merge GB/s (algorithmic bytes / time)"
    unit = "GB/s"
    K = 8
    launches_per_step = 1

    def __init__(self, rank, world, device):
        super().__init__(rank, world, device)
        self.shapes = synth.roberta_shapes()
        self.d = synth.total_numel(self.shapes)
        self.bytes_per_step = (self.K + 2) * self.d * 4

    def config(self):
        return {"workload": "BLaIR-base (RoBERTa-base, d=124,645,632, P=199) K=8 per-layer lambda merge (G=13) "
                            "from stored task vectors; merge half of BASELINE config 2",
                "K": self.K, "d": self.d, "G": 13, "l2": "inputs (4.5 GB) exceed L2, no flush needed",
                "parallelism": "single GPU (one merge is a few ms; the multi-GPU form is --workload ties_sharded)"}

    # -- device-resident arm
    def setup(self):
        from mergerec_b200.merger.algorithms import get_task_vectors
        from mergerec_b200.merger.layout import FlatLayout
        g = torch.Generator(device=self.device).manual_seed(1234 + self.rank)
        d, K = self.d, self.K
        self.base = torch.randn(d, generator=g, device=self.device) * 0.02
        self.models = [self.base + 1e-3 * torch.randn(d, generator=g, device=self.device) for _ in range(K)]
        self.T = get_task_vectors(self.base, self.models)
        self.rows = list(self.T.unbind(0))
        self.layout = FlatLayout.from_shape_dict(self.shapes)
        self.seg_end, self.seg_group, keys = self.layout.device_blocks(True, self.device)
        rng = np.random.Generator(np.random.PCG64(5))
        self.w = torch.from_numpy(rng.uniform(0.1, 0.5, size=(len(keys), K)).astype(np.float32)).to(self.device)
        self.out = torch.empty(d, dtype=torch.float32, device=self.device)

    def step(self):
        from mergerec_b200 import _lib
        from mergerec_b200.merger.algorithms._common import merge_axpy
        merge_axpy(self.base, self.rows, self.w, _lib.MR_ORDER_SUM_FIRST, False, self.seg_end, self.seg_group, out=self.out)

    def outputs(self):
        return {"merged": _output(self.out)}

    def units_per_step_all_ranks(self):
        return self.bytes_per_step / GB     # one job; with several ranks every rank repeats it (no "x N" credit)

    # -- end-to-end arm: pinned host flat vectors in, merged flat vector out
    def setup_e2e(self):
        self.h_base = _pinned(self.base.cpu())
        self.h_T = _pinned(self.T.cpu())
        self.h_out = torch.empty(self.d, dtype=torch.float32, pin_memory=True)
        self.h2d_bytes = (self.K + 1) * self.d * 4
        self.d2h_bytes = self.d * 4

    def step_e2e(self):
        self.base.copy_(self.h_base, non_blocking=True)
        self.T.copy_(self.h_T, non_blocking=True)
        self.step()
        self.h_out.copy_(self.out, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    # -- roofline of the dominant kernel (the only one here)
    def roofline(self, peaks):
        from bench import event_time_ms
        ms = event_time_ms(self.step, 20)
        achieved = self.bytes_per_step / GB / (ms * 1e-3)
        return _with_traffic({"bound": "hbm", "kernel": "mr::merge_kernel<8, SUM_FIRST, segmented, vec4>", "achieved": achieved,
                "peak": peaks["hbm_gbs"], "peak_source": peaks["source"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": None, "ms_per_launch": ms,
                "algorithmic_bytes_per_launch": self.bytes_per_step}, "merge_kernel")

    # -- CPU arms (oracle port of the reference algorithm)
    def _cpu_inputs(self, d):
        rng = np.random.Generator(np.random.PCG64(7))
        base = rng.standard_normal(d, dtype=np.float32) * np.float32(0.02)
        T = rng.standard_normal((self.K, d), dtype=np.float32) * np.float32(1e-3)
        from oracle import oracle as orc
        sb, se, sg, keys = orc.segment_table(self.shapes, layer_wise=True)
        w = rng.uniform(0.1, 0.5, size=(len(keys), self.K)).astype(np.float32)
        return base, T, w, sb, se, sg

    def _cpu_time(self, reps):
        from oracle import oracle as orc
        base, T, w, sb, se, sg = self._cpu_inputs(self.d)
        orc.lambda_merge(base, T, w, sb, se, sg)
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            orc.lambda_merge(base, T, w, sb, se, sg)
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts)), orc.max_threads()

    def cpu_baseline(self):
        t, cores = self._cpu_time(3)
        return {"value": self.bytes_per_step / GB / t, "unit": self.unit, "cores": cores, "kind": "port",
                "sample": f"full workload (d={self.d}, K={self.K}), median of 3 after 1 warm-up, OpenMP C oracle",
                "seconds_per_step": t}

    def reference_arm(self, steps, warmup):
        t, cores = self._cpu_time(max(1, steps))
        return {"value": self.bytes_per_step / GB / t, "ms_per_step": t * 1e3, "cores": cores,
                "sample": f"full workload (d={self.d}, K={self.K}) per step, OpenMP C oracle port"}


class TiesCfg2(LambdaMergeK8):
    """BASELINE config 2: TIES merge (trim 20 %, sign election, disjoint mean) of 8 BLaIR-base domain models with
    per-layer lambda.  One step = the reference-shaped pipeline `get_ties_vectors(density=0.2)` (A6-A8) followed
    by the layer-wise lambda merge (A4).  Algorithmic bytes per step: (2K+1)*d*4 + (K+2)*d*4."""

    name = "ties_cfg2"
    launches_per_step = 15  # own kernels: init, 2 x (sample pass, pick), mid, spec pass, 2 x (cand_hist, pick), compact, final, patch, merge

    def __init__(self, rank, world, device):
        super().__init__(rank, world, device)
        self.bytes_build = (2 * self.K + 1) * self.d * 4
        self.bytes_merge = (self.K + 2) * self.d * 4
        self.bytes_per_step = self.bytes_build + self.bytes_merge

    def config(self):
        return {"workload": "BASELINE config 2: TIES merge (density 0.2, global trim, sign election, disjoint mean) "
                            "of K=8 BLaIR-base (RoBERTa-base, d=124,645,632, P=199) domain models + per-layer "
                            "lambda merge (G=13)",
                "K": self.K, "d": self.d, "G": 13, "density": 0.2,
                "l2": "inputs (4.5 GB) exceed L2, no flush needed",
                "select_status": "checked on the host after the timed loop (stream-ordered step)",
                "parallelism": "single GPU (one merge is a few ms; the multi-GPU form is --workload ties_sharded)"}

    def setup(self):
        super().setup()
        from mergerec_b200.merger.layout import alloc_rows
        self.That = alloc_rows(self.K, self.d, self.device)
        self.Trows = list(self.That.unbind(0))
        del self.T, self.rows
        self._status = None
        self._try_capture()

    def _eager_step(self, defer=True):
        """select -> build -> per-layer merge, stream-ordered: the select's status word is checked by the host after
        the timed loop (`finish`), not between the kernels (`defer=False` is the public API's immediate check)."""
        from mergerec_b200 import _lib
        from mergerec_b200.merger.algorithms import ties as T
        from mergerec_b200.merger.algorithms._common import merge_axpy
        if os.environ.get("MR_BENCH_TIES_TWO_PASS"):      # round-1 pipeline: select (one full pass), then build (another)
            if defer:
                cut, self._status = T.select_kth_largest(self.base, self.models, int(0.2 * self.d), None, defer_status=True)
            else:
                cut = T.ties_select(self.base, self.models, 0.2)
            T._build(self.base, self.models, cut, _lib.MR_TIES_VECTORS, out=self.That, ldo=self.That.stride(0))
        elif defer:
            _, self._status = T.select_build(self.base, self.models, int(0.2 * self.d), _lib.MR_TIES_VECTORS, self.That,
                                             ldo=self.That.stride(0), defer_status=True)
        else:
            T.select_build(self.base, self.models, int(0.2 * self.d), _lib.MR_TIES_VECTORS, self.That, ldo=self.That.stride(0))
        merge_axpy(self.base, self.Trows, self.w, _lib.MR_ORDER_SUM_FIRST, False, self.seg_end, self.seg_group, out=self.out)

    def _try_capture(self):
        """One CUDA graph for the whole step (12 launches of this package, all stream-ordered)."""
        self.graph = None
        if os.environ.get("MR_BENCH_NO_GRAPH"):
            return
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    self._eager_step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._eager_step()
            g.replay()
            torch.cuda.synchronize()
            self.finish()
            self.graph = g
        except Exception as e:  # noqa: BLE001 -- report, keep the eager path
            print(f"[ties_cfg2] CUDA graph capture unavailable ({type(e).__name__}: {e}); eager launches", file=__import__("sys").stderr)
            self.graph = None
            torch.cuda.synchronize()

    def step(self):
        if getattr(self, "graph", None) is not None:
            self.graph.replay()
        else:
            self._eager_step()

    def finish(self):
        """After a timed loop: the deferred status of the last select (every step ran the same inputs)."""
        from mergerec_b200.merger.algorithms import ties as T
        if getattr(self, "_status", None) is not None:
            T.verify_select_status(self._status)

    def step_fused(self):
        from mergerec_b200.merger.algorithms import ties as T
        T.merge_ties_lambda(self.base, self.models, 0.2, self.w, self.seg_end, self.seg_group, out=self.out)

    def setup_e2e(self):
        self.h_base = _pinned(self.base.cpu())
        self.h_models = [_pinned(m.cpu()) for m in self.models]
        self.h_out = torch.empty(self.d, dtype=torch.float32, pin_memory=True)
        self.h2d_bytes = (self.K + 1) * self.d * 4
        self.d2h_bytes = self.d * 4

    def step_e2e(self):
        self.base.copy_(self.h_base, non_blocking=True)
        for m, h in zip(self.models, self.h_models):
            m.copy_(h, non_blocking=True)
        self._e2e_kernels()
        self.h_out.copy_(self.out, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def _e2e_kernels(self):
        self._eager_step(defer=False)      # the public get_ties_vectors path: status checked on the host right away

    def roofline(self, peaks):
        from bench import event_time_ms
        from mergerec_b200 import _lib
        from mergerec_b200.merger.algorithms import ties as T
        cut = T.ties_select(self.base, self.models, 0.2)
        lib = _lib.load()
        K, d = self.K, self.d
        ws_bytes = int(lib.mr_ties_workspace_bytes(d, K))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
        cut2 = torch.empty(K, dtype=torch.int64, device=self.device)
        status = torch.zeros(K, dtype=torch.int32, device=self.device)
        parr = _lib.ptr_array(self.models)

        def select():
            _lib.check(lib.mr_ties_select(_lib.dptr(self.base), parr, K, d, None, int(0.2 * d), _lib.dptr(cut2),
                                          _lib.dptr(status), _lib.dptr(ws), ws_bytes, _lib.stream_handle()), "select")

        def build():
            T._build(self.base, self.models, cut, _lib.MR_TIES_VECTORS, out=self.That, ldo=self.That.stride(0))

        # lambda-gradient reduction (A5; the backward kernel of BASELINE config 3) against the same K x d rows
        from mergerec_b200.merger.weight_learning.module._base import _lambda_grad
        grad = torch.randn(self.d, device=self.device)
        seg_off, seg_len = self.layout.device_segments(self.device)
        grads = [grad[o:o + n] for o, n in zip(seg_off.tolist(), seg_len.tolist())]
        lgrad = lambda: _lambda_grad(grads, self.layout, self.That, self.seg_group, int(self.w.shape[0]))  # noqa: E731
        lgrad()
        ms_lgrad = event_time_ms(lgrad, 5)
        lgrad_bytes = (K + 1) * d * 4
        del grad, grads

        def one_pass():
            T.select_build(self.base, self.models, int(0.2 * d), _lib.MR_TIES_VECTORS, self.That, ldo=self.That.stride(0), defer_status=True)

        ms_build = event_time_ms(build, 10)
        ms_select = event_time_ms(select, 10)
        ms_onepass = event_time_ms(one_pass, 10)
        ms_merge = event_time_ms(self._merge_only, 10)
        ms_fused = event_time_ms(self.step_fused, 5)
        ach = self.bytes_build / GB / (ms_onepass * 1e-3)
        sel_bytes = (K + 1) * d * 4
        return _with_traffic({"bound": "hbm", "kernel": "mr::ties_spec_kernel<8, VECTORS, vec4> + sample passes + exact-cut finish + fix-up "
                                                        "(get_ties_vectors in one pass over the data: mr_ties_select_build)",
                "achieved": ach, "peak": peaks["hbm_gbs"], "peak_source": peaks["source"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "traffic": None, "ms_per_launch": ms_onepass,
                "algorithmic_bytes_per_launch": self.bytes_build,
                "other_kernels": {
                    "two-pass pipeline, select only (sample + 1 full pass + finish)": {"ms": ms_select, "GB/s": sel_bytes / GB / (ms_select * 1e-3), "bytes": sel_bytes},
                    "two-pass pipeline, build only (ties_build_kernel<8, VECTORS, vec4>)": {"ms": ms_build, "GB/s": self.bytes_build / GB / (ms_build * 1e-3), "bytes": self.bytes_build},
                    "lambda-gradient reduction (lambda_grad_kernel, incl. host pointer-table upload)": {"ms": ms_lgrad, "GB/s": lgrad_bytes / GB / (ms_lgrad * 1e-3), "bytes": lgrad_bytes},
                    "lambda merge (merge_kernel)": {"ms": ms_merge, "GB/s": self.bytes_merge / GB / (ms_merge * 1e-3), "bytes": self.bytes_merge},
                    "fused TIES + lambda merge in one pass, That never materialised (merge_ties_lambda)": {"ms": ms_fused, "GB/s": self.bytes_merge / GB / (ms_fused * 1e-3), "bytes": self.bytes_merge},
                }}, "ties_spec_kernel")

    def extra(self):
        return {"cuda_graph": getattr(self, "graph", None) is not None}

    def _merge_only(self):
        from mergerec_b200 import _lib
        from mergerec_b200.merger.algorithms._common import merge_axpy
        merge_axpy(self.base, self.Trows, self.w, _lib.MR_ORDER_SUM_FIRST, False, self.seg_end, self.seg_group, out=self.out)

    # -- CPU arms.  Port: the OpenMP C oracle at the FULL size of the workload (about 2 s per step).  Reference: the
    #    unmodified `get_ties_vectors` + `TaskVectorMergingModuleLayerWise._merge_task_vectors` from baseline/_ref on a
    #    RoBERTa-shaped slice (12 layers, hidden 64: same P = 199 tensors and G = 13 groups, d = 3.85 M) -- at full
    #    size the reference needs minutes per step (single-threaded torch.topk over 1.2e8 elements per model).
    def _port_inputs(self):
        rng = np.random.Generator(np.random.PCG64(7))
        d = self.d
        base = rng.standard_normal(d, dtype=np.float32) * np.float32(0.02)
        models = [base + np.float32(1e-3) * rng.standard_normal(d, dtype=np.float32) for _ in range(self.K)]
        from oracle import oracle as orc
        sb, se, sg, keys = orc.segment_table(self.shapes, layer_wise=True)
        w = rng.uniform(0.1, 0.5, size=(len(keys), self.K)).astype(np.float32)
        return base, models, w, sb, se, sg

    def _port_step_fn(self):
        from oracle import oracle as orc
        base, models, w, sb, se, sg = self._port_inputs()

        def step():
            That = orc.ties_vectors(base, models, 0.2)
            orc.lambda_merge(base, That, w, sb, se, sg)
        return step, self.bytes_per_step, (f"full workload (d={self.d}, K={self.K}): ties_vectors + per-layer lambda merge, "
                                           "OpenMP C oracle port")

    def _reference_step_fn(self):
        ref = reference_package()
        if ref is None:
            return None
        from rec_retrieval.merger.algorithms.ties import get_ties_vectors
        from rec_retrieval.merger.weight_learning.module.layer_wise import TaskVectorMergingModuleLayerWise
        shapes = synth.roberta_shapes(hidden=64, ffn=256)
        d = synth.total_numel(shapes)
        g = torch.Generator().manual_seed(7)
        base = torch.randn(d, generator=g) * 0.02
        models = [base + 1e-3 * torch.randn(d, generator=g) for _ in range(self.K)]
        shape_dict = {k: torch.Size(v) for k, v in shapes.items()}

        class _NoModel(torch.nn.Module):
            def forward(self, x):
                return x

        def step():
            That = get_ties_vectors(base, models, 0.2)
            mod = TaskVectorMergingModuleLayerWise(base, That, _NoModel(), shape_dict, disable_softmax=True)
            with torch.no_grad():
                mod._merge_task_vectors()
        nbytes = ((2 * self.K + 1) + (self.K + 2)) * d * 4
        return step, nbytes, (f"UNMODIFIED reference (get_ties_vectors + TaskVectorMergingModuleLayerWise._merge_task_vectors) on a "
                              f"RoBERTa-shaped slice: 12 layers, hidden 64, P=199, G=13, d={d}, K={self.K}, density 0.2")

    def cpu_baseline(self):
        from oracle import oracle as orc
        fn, nbytes, sample = self._port_step_fn()
        t, ts = timed_steps(fn, 3, 1)
        t = float(np.median(ts))
        out = {"value": nbytes / GB / t, "unit": self.unit, "cores": orc.max_threads(), "kind": "port",
               "sample": sample + "; median of 3 after 1 warm-up", "seconds_per_step": t}
        r = self._reference_step_fn()
        if r is not None:
            rfn, rbytes, rsample = r
            rt, rts = timed_steps(rfn, 2, 1)
            rt = float(np.median(rts))
            out["reference"] = {"value": rbytes / GB / rt, "unit": self.unit, "cores": torch.get_num_threads(), "kind": "reference",
                                "sample": rsample + "; median of 2 after 1 warm-up", "seconds_per_step": rt}
        return out

    def reference_arm(self, steps, warmup):
        from oracle import oracle as orc
        r = self._reference_step_fn()
        if r is not None:
            fn, nbytes, sample = r
            t, _ = timed_steps(fn, steps, warmup)
            return {"value": nbytes / GB / t, "ms_per_step": t * 1e3, "cores": torch.get_num_threads(), "kind": "reference",
                    "sample": sample + " per step"}
        fn, nbytes, sample = self._port_step_fn()
        t, _ = timed_steps(fn, steps, warmup)
        return {"value": nbytes / GB / t, "ms_per_step": t * 1e3, "cores": orc.max_threads(), "kind": "port",
                "sample": sample + " per step"}


class EvalCatalog(Workload):
    """BASELINE config 5 (evaluator): full-catalog scoring of Q query embeddings against an N-item table (E = 768),
    fused per-row top-100, label rank and Recall/NDCG.  The item table is sharded over the ranks (N / world rows
    each, strong scaling); every rank scores all queries against its shard, the per-rank top-K lists are exchanged by
    ONE NCCL all-gather and merged.  One step = one pass of all Q queries over the whole catalog.

    Default sizes are config 5 itself: Q = 65,536 queries, N = 1,000,000 items, E = 768, top-100 (1.0e14 logical FLOP,
    x3 tensor passes); MR_BENCH_EVAL_Q / _N / _K / _E override them (for debugging only)."""

    name = "eval_cfg5"
    label = "BASELINE config 5"
    metric = "catalog scores/sec (Q*N / time, fused scoring + top-K + Recall/NDCG)"
    unit = "scores/s"
    dtype = "tf32x3 (fp32-faithful split, fp32 accumulate)"
    scaling = "strong"
    e2e_steps_cap = 3
    sizes = dict(Q=65536, N=1_000_000, E=768, K=100)
    ks_low = 10
    cpu_sample = dict(Q=128)          # queries per CPU step (full catalog width)
    accuracy_rows = 2048

    def __init__(self, rank, world, device):
        super().__init__(rank, world, device)
        self.Q = int(os.environ.get("MR_BENCH_EVAL_Q", self.sizes["Q"]))
        self.N = int(os.environ.get("MR_BENCH_EVAL_N", self.sizes["N"]))
        self.E = int(os.environ.get("MR_BENCH_EVAL_E", self.sizes["E"]))
        self.K = int(os.environ.get("MR_BENCH_EVAL_K", self.sizes["K"]))
        self.mode = int(os.environ.get("MR_BENCH_EVAL_MODE", 0))
        self.ks = sorted({min(self.ks_low, self.K), self.K})
        self.flops = 2.0 * self.Q * self.N * self.E
        self.l2_flush = (self.Q + self.N) * self.E * 8 < (256 << 20)   # hi + lo operands smaller than 2x L2: flush
        # split is part of the operand format (prepared once); per step: score_topk, its list merge, [all-gather is
        # NCCL's], shard merge, label_rank
        self.launches_per_step = 3 if world == 1 else 4
        self._stage = None
        self._checksum = None
        self._accuracy = None

    def companion(self):
        return TiesCfg2 if self.world == 1 else TiesSharded

    def config(self):
        return {"workload": f"{self.label}: {self.Q} query seqs x {self.N}-item catalog, E={self.E}, "
                            f"top-{self.K}, Recall/NDCG@{{{','.join(str(k) for k in self.ks)}}}; item table row-sharded over the GPUs, "
                            "one NCCL all-gather of the per-GPU top-K lists + merge",
                "Q": self.Q, "N": self.N, "E": self.E, "K": self.K, "mode": "tf32x3" if self.mode == 0 else "tf32x1",
                "l2": ("operands fit L2: a 512 MB buffer is written between timed steps (flush)" if self.l2_flush else
                       f"item table ({self.N * self.E * 8 / 1e9:.1f} GB as hi/lo operands) exceeds L2, no flush needed"),
                "parallelism": "item table sharded N/G rows per GPU, queries replicated (strong scaling)"}

    # ---------------------------------------------------------------------------------------------- inputs
    def _make_inputs(self, device, lo, hi):
        """Same queries / labels on every rank; the item table generated chunk by chunk (seeded per chunk) so that every
        rank sees the same catalog and keeps rows [lo, hi).  Half of the queries are planted near their label item so
        Recall / NDCG are non-trivial."""
        g = torch.Generator(device=device).manual_seed(99)
        users = torch.randn(self.Q, self.E, generator=g, device=device)
        labels = torch.randint(0, self.N, (self.Q,), generator=g, device=device)
        planted = torch.rand(self.Q, generator=g, device=device) < 0.5
        items = torch.empty(hi - lo, self.E, device=device)
        label_rows = torch.empty(self.Q, self.E, device=device)
        chunk = 65536
        for c0 in range(0, self.N, chunk):
            c1 = min(self.N, c0 + chunk)
            gi = torch.Generator(device=device).manual_seed(1000 + c0 // chunk)
            rows = torch.nn.functional.normalize(torch.randn(c1 - c0, self.E, generator=gi, device=device), dim=-1)
            a, b = max(c0, lo), min(c1, hi)
            if a < b:
                items[a - lo:b - lo] = rows[a - c0:b - c0]
            sel = (labels >= c0) & (labels < c1)
            if bool(sel.any()):
                label_rows[sel] = rows[labels[sel] - c0]
        users = torch.where(planted[:, None], label_rows + 0.5 * users / self.E ** 0.5, users)
        return torch.nn.functional.normalize(users, dim=-1), items, labels

    def setup(self):
        import torch.distributed as dist
        from mergerec_b200.evaluator import Evaluator, ShardedItemTable, shard_bounds
        lo, hi = shard_bounds(self.N, self.world, self.rank)
        self.users, self.items, self.labels = self._make_inputs(self.device, lo, hi)
        self.lo = lo
        self.group = dist.group.WORLD if self.world > 1 else None
        self.table = ShardedItemTable(self.items, id_base=lo, n_total=self.N, group=self.group)
        self.ev = Evaluator(["RECALL", "NDCG"], self.ks)
        self.queries = self.ev.prepare_queries(self.users)      # operand format of the kernel: split once, reused
        self.last = None

    def step(self):
        self.last = self.ev.evaluate_embeddings(self.queries, self.table, self.labels, mode=self.mode)

    def outputs(self):
        return {name: np.float64(v) for name, v in self.last.items()}

    def units_per_step_all_ranks(self):
        return float(self.Q) * float(self.N)

    # ---------------------------------------------------------------------------------------------- after the loop
    def finish(self):
        """Every rank: (1) checksums of the merged top-K lists -- integers that must not depend on the number of GPUs;
        (2) the step cut into stages with CUDA events / host clocks (where the non-kernel time goes)."""
        import torch.distributed as dist
        from mergerec_b200.evaluator.evaluator import score_topk
        from mergerec_b200.evaluator.metrics import label_rank
        from mergerec_b200.evaluator.sharded import exchange_packed, new_packed_list
        vals, ids = self.ev.topk_embeddings(self.queries, self.table, self.K, mode=self.mode)
        pos = torch.arange(1, self.K + 1, device=self.device, dtype=torch.int64)
        self._checksum = {
            "topk_ids": int(((ids.to(torch.int64) + 1) * pos).sum().item()),
            "topk_score_bits": int((vals.view(torch.int32).to(torch.int64) * pos).sum().item()),
            "note": "sum over (q, r) of (id + 1) * (r + 1) and of score bits * (r + 1): equal for every --gpus N"}
        del vals, ids

        def ev_ms(fn, reps=3):
            fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            b.synchronize()
            return a.elapsed_time(b) / reps

        Q, K = self.Q, self.K
        local, lv, li = new_packed_list(Q, K, self.device)
        st = {"score_topk_kernel_plus_split_merge": ev_ms(lambda: score_topk(self.queries.hi, self.queries.lo, self.table, K, self.mode, out=(lv, li)), 2)}
        if self.world > 1:
            gathered = self.table.gather_buffer(Q, K)
            dist.barrier()
            st["all_gather_plus_shard_merge"] = ev_ms(lambda: exchange_packed(local, K, self.group, gathered=gathered))
            st["all_gather_alone"] = ev_ms(lambda: dist.all_gather_into_tensor(gathered.view(self.world * 2 * Q, K), local.view(2 * Q, K), group=self.group))
            ids = exchange_packed(local, K, self.group, gathered=gathered)[1]
        else:
            ids = li
        st["label_rank_kernel"] = ev_ms(lambda: label_rank(ids, self.labels))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            self.ev.metrics_from_ids(ids, self.labels)
        st["label_rank_d2h_and_host_metrics_wall"] = (time.perf_counter() - t0) / 3 * 1e3
        if self.world > 1:
            t = torch.tensor([st[k] for k in sorted(st)], dtype=torch.float64, device=self.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            st = {k: float(v) for k, v in zip(sorted(st), t.tolist())}
        self._stage = st

    # ---------------------------------------------------------------------------------------------- end to end
    def setup_e2e(self):
        self.h_users = _pinned(self.users.cpu())
        self.h_items = _pinned(self.items.cpu())
        self.h_labels = _pinned(self.labels.cpu())
        self.h2d_bytes = -(-self.h_users.shape[0] // self.world) * self.E * 4 + self.h_items.numel() * 4 + self.h_labels.numel() * 8
        self.d2h_bytes = self.Q * 4          # the rank of each label; the metric floats are finished on the host

    def step_e2e(self):
        """Host embeddings in, metric floats out, through the public API for host-resident catalogs
        (`Evaluator.evaluate_embeddings_streamed`): H2D of the queries and labels, then this rank's item rows in
        geometrically growing chunks on a copy stream while the previous chunk is split and scored, merge of the chunk
        lists, exchange, label rank, D2H of the ranks, host finalisation."""
        from mergerec_b200.evaluator import replicate_from_host
        users = replicate_from_host(self.h_users, self.group)      # 1/N of the queries per rank over PCIe, all-gather over NVLink
        labels = self.h_labels.to(self.device, non_blocking=True)
        self.last = self.ev.evaluate_embeddings_streamed(users, self.h_items, labels, id_base=self.lo, n_total=self.N,
                                                         group=self.group, mode=self.mode)

    def teardown_e2e(self):
        del self.h_users, self.h_items, self.h_labels

    # ---------------------------------------------------------------------------------------------- roofline
    def roofline(self, peaks):
        from bench import event_time_ms, measure_tf32_peak
        from mergerec_b200.evaluator.evaluator import score_topk
        ms = event_time_ms(lambda: score_topk(self.queries.hi, self.queries.lo, self.table, self.K, self.mode), 2)
        passes = 3 if self.mode == 0 else 1
        local_flops = 2.0 * self.Q * self.table.n_local * self.E
        ach = passes * local_flops / (ms * 1e-3) / 1e12
        # There is no TF32 entry in MEASURED_PEAKS.json, so the denominator is the LARGEST dense-TF32 rate this run can
        # vouch for: cuBLAS TF32 GEMMs measured here (burst = best of 10; sustained = back to back at the 1 kW power cap)
        # and the bf16 peaks of MEASURED_PEAKS.json halved.  (Rounds 1-2 switched between burst and sustained by launch
        # length; since the item-stream pacing this kernel draws less DRAM power than cuBLAS and overtook the sustained
        # figures, so the conservative choice is the maximum.)  All four fractions are listed below.
        tf32 = measure_tf32_peak(self.device)
        cands = {"cuBLAS TF32 GEMM 8192^3 measured in this run, burst (best of 10)": tf32["tf32_tflops"],
                 "cuBLAS TF32 GEMM 8192^3 measured in this run, sustained (back to back for ~2 s)": tf32["tf32_tflops_sustained"],
                 "MEASURED_PEAKS.json bf16 burst / 2": peaks["bf16_tflops"] / 2,
                 "MEASURED_PEAKS.json bf16 sustained / 2": peaks["bf16_tflops_sustained"] / 2}
        peak_name = max(cands, key=cands.get)
        peak = cands[peak_name]
        roof = {"bound": "tensor", "kernel": "mr::st::score_topk_kernel<2, 32> (tcgen05.mma kind::tf32, cta_group::2) + list merge",
                "achieved": ach, "peak": peak,
                "peak_source": "largest of the four dense-TF32 candidates: " + peak_name,
                "unit": "TFLOP/s", "frac": ach / peak, "traffic": None, "ms_per_launch": ms,
                "tensor_passes": passes, "logical_tflops": local_flops / (ms * 1e-3) / 1e12,
                "algorithmic_flops_per_launch": passes * local_flops,
                "tf32_peak_measured": tf32,
                "frac_of_measured_burst": ach / tf32["tf32_tflops"], "frac_of_measured_sustained": ach / tf32["tf32_tflops_sustained"],
                "frac_of_bf16_derived_burst": ach / (peaks["bf16_tflops"] / 2),
                "frac_of_bf16_derived_sustained": ach / (peaks["bf16_tflops_sustained"] / 2)}
        if self.world == 1 and (self.Q, self.N, self.E, self.K) == (65536, 1_000_000, 768, 100):
            roof = _with_traffic(roof, "score_topk_kernel")     # the committed ncu capture is of exactly this launch
        if self.world == 1 and not os.environ.get("MR_BENCH_SKIP_ACCURACY"):
            try:
                self._accuracy = self.accuracy()
            except Exception as e:  # noqa: BLE001 -- the accuracy figure is reported, never fatal
                self._accuracy = {"error": repr(e)}
        return roof

    def accuracy(self):
        """Parity figure of the 3xTF32 path AT THIS SCALE on Gaussian (non-grid) inputs: the top-K of a slice of the
        queries against the whole catalog, compared with (a) plain fp32 CUDA-core scoring (`mr_scores_fp32`: one fp32
        FMA chain per score) + `mr_topk_rows` and (b) an fp64 ranking (torch fp64 matmul + stable sort by
        (score desc, id asc))."""
        from mergerec_b200 import _lib
        from mergerec_b200.evaluator.evaluator import topk_rows
        from mergerec_b200.evaluator.metrics import label_rank, ndcg_from_ranks, recall_from_ranks
        lib = _lib.load()
        Qs, K, N, E = min(self.accuracy_rows, self.Q), self.K, self.table.n_local, self.E
        users = self.users[:Qs].contiguous()
        v3, i3 = self.ev.topk_embeddings(users, self.table, K, mode=self.mode)
        # (a) fp32 CUDA-core scores, materialised in row chunks
        i32 = torch.empty((Qs, K), dtype=torch.int32, device=self.device)
        v32 = torch.empty((Qs, K), dtype=torch.float32, device=self.device)
        i64 = torch.empty((Qs, K), dtype=torch.int32, device=self.device)
        v64 = torch.empty((Qs, K), dtype=torch.float64, device=self.device)
        rows = max(1, min(Qs, (8 << 30) // (N * 8)))
        items64 = self.items.double()
        for q0 in range(0, Qs, rows):
            q1 = min(Qs, q0 + rows)
            sc = torch.empty((q1 - q0, N), dtype=torch.float32, device=self.device)
            _lib.check(lib.mr_scores_fp32(_lib.dptr(users[q0:q1]), q1 - q0, _lib.dptr(self.items), N, E, _lib.dptr(sc), N,
                                          _lib.stream_handle()), "mr_scores_fp32")
            v, i = topk_rows(sc, K)
            v32[q0:q1], i32[q0:q1] = v, i
            del sc
            s64 = users[q0:q1].double() @ items64.T
            v, i = torch.topk(s64, K + 8, dim=1)                 # a few extra, then the canonical order among equal scores
            order = torch.argsort(i, dim=1, stable=True)
            v, i = torch.gather(v, 1, order), torch.gather(i, 1, order)
            order = torch.argsort(v, dim=1, descending=True, stable=True)
            v, i = torch.gather(v, 1, order)[:, :K], torch.gather(i, 1, order)[:, :K]
            v64[q0:q1], i64[q0:q1] = v, i.to(torch.int32)
            del s64
        del items64

        def cmp_ids(a, b):
            diff = a != b
            rows_diff = diff.any(dim=1)
            first = torch.where(rows_diff, diff.to(torch.int32).argmax(dim=1), torch.full_like(rows_diff, K, dtype=torch.int64))
            same_set = (torch.sort(a, dim=1).values == torch.sort(b, dim=1).values).all(dim=1)
            return {"rows_differing": int(rows_diff.sum()), "rows": int(a.shape[0]),
                    "first_differing_rank_min": int(first.min()) if bool(rows_diff.any()) else None,
                    "rows_with_different_id_SET": int((~same_set).sum())}

        labels = self.labels[:Qs]

        def mets(ids):
            r = label_rank(ids, labels).cpu().numpy()
            return {f"Recall@{k}": recall_from_ranks(r, k) for k in self.ks} | {f"NDCG@{k}": ndcg_from_ranks(r, k) for k in self.ks}

        m3, m32, m64 = mets(i3), mets(i32), mets(i64)
        # smallest fp64 gap between neighbours of the fp64 list: what a swap has to overcome
        gaps = (v64[:, :-1] - v64[:, 1:])
        res = {"slice": f"first {Qs} queries x all {N} items, top-{K}, unit-norm Gaussian embeddings (half of the queries planted near their label)",
               "tf32x3_vs_fp64": cmp_ids(i3, i64), "tf32x3_vs_fp32_cuda_cores": cmp_ids(i3, i32), "fp32_cuda_cores_vs_fp64": cmp_ids(i32, i64),
               "max_abs_score_error_vs_fp64_at_equal_ids": {
                   "tf32x3": float(((v3.double() - v64).abs() * (i3 == i64)).max()),
                   "fp32_cuda_cores": float(((v32.double() - v64).abs() * (i32 == i64)).max())},
               "fp64_neighbour_gap": {"min": float(gaps.min()), "median": float(gaps.median())},
               "metrics_tf32x3": m3, "metrics_fp32": m32, "metrics_fp64": m64,
               "metrics_identical_to_fp64": m3 == m64, "metrics_identical_to_fp32": m3 == m32}
        return res

    def extra(self):
        out = {"metrics": self.last, "checksum": self._checksum, "stage_ms": self._stage}
        if self._accuracy is not None:
            out["accuracy"] = self._accuracy
        return out

    # ---------------------------------------------------------------------------------------------- CPU arms
    # One CPU step = `cpu_sample["Q"]` queries against the WHOLE catalog: scores = U @ I.T (module.py:137) followed by
    # Evaluator(["RECALL", "NDCG"], ks)(scores, labels) (evaluator.py:31-49).  Reference = the unmodified
    # rec_retrieval.evaluator from baseline/_ref (torch CPU matmul + torch.topk + the python metric loops); port = numpy
    # BLAS sgemm + the OpenMP C top-K + python metric loops of oracle/.
    def _cpu_inputs(self):
        Qs = min(self.Q, self.cpu_sample["Q"])
        rng = np.random.Generator(np.random.PCG64(7))
        users = rng.standard_normal((Qs, self.E), dtype=np.float32)
        items = rng.standard_normal((self.N, self.E), dtype=np.float32)
        labels = rng.integers(0, self.N, size=Qs)
        return users, items, labels, Qs

    def _port_step_fn(self):
        from oracle import oracle as orc
        users, items, labels, Qs = self._cpu_inputs()
        ks = [min(k, self.N) for k in self.ks]

        def step():
            scores = orc.scores_f32(users, items)
            orc.evaluate(scores, labels, ["RECALL", "NDCG"], ks)
        return step, float(Qs) * self.N, (f"{Qs} queries x the whole {self.N}-item catalog (E={self.E}), top-{ks[-1]}: numpy/BLAS sgemm + "
                                          "OpenMP C top-K + python metric loops (oracle port)")

    def _reference_step_fn(self):
        if reference_package() is None:
            return None
        from rec_retrieval.evaluator import Evaluator as RefEvaluator
        users, items, labels, Qs = self._cpu_inputs()
        tu, ti, tl = torch.from_numpy(users), torch.from_numpy(items), torch.from_numpy(labels)
        ev = RefEvaluator(["RECALL", "NDCG"], [min(k, self.N) for k in self.ks])

        def step():
            scores = tu @ ti.T
            ev(scores, tl)
        return step, float(Qs) * self.N, (f"UNMODIFIED reference: scores = U @ I.T (torch CPU fp32) + rec_retrieval.evaluator.Evaluator on "
                                          f"{Qs} queries x the whole {self.N}-item catalog (E={self.E}), top-{self.ks[-1]}")

    def cpu_baseline(self):
        from oracle import oracle as orc
        fn, units, sample = self._port_step_fn()
        _, ts = timed_steps(fn, 3, 1)
        t = float(np.median(ts))
        port = {"value": units / t, "unit": self.unit, "cores": max(orc.max_threads(), torch.get_num_threads()), "kind": "port",
                "sample": sample + "; median of 3 after 1 warm-up", "seconds_per_step": t}
        r = self._reference_step_fn()
        if r is None:
            return port
        rfn, runits, rsample = r
        _, rts = timed_steps(rfn, 3, 1)
        rt = float(np.median(rts))
        return {"value": runits / rt, "unit": self.unit, "cores": torch.get_num_threads(), "kind": "reference",
                "sample": rsample + "; median of 3 after 1 warm-up", "seconds_per_step": rt, "port": port}

    def reference_arm(self, steps, warmup):
        from oracle import oracle as orc
        r = self._reference_step_fn()
        if r is not None:
            fn, units, sample = r
            t, _ = timed_steps(fn, steps, warmup)
            return {"value": units / t, "ms_per_step": t * 1e3, "cores": torch.get_num_threads(), "kind": "reference",
                    "sample": sample + " per step"}
        fn, units, sample = self._port_step_fn()
        t, _ = timed_steps(fn, steps, warmup)
        return {"value": units / t, "ms_per_step": t * 1e3, "cores": max(orc.max_threads(), torch.get_num_threads()), "kind": "port",
                "sample": sample + " per step"}


class CollabStepCfg3(Workload):
    """BASELINE config 3: one MergeRec collaborative-merging optimisation step at K = 8 BLaIR-base (RoBERTa-base)
    domains -- layer-wise lambda merge (A4) into one flat buffer whose slices become the encoder's parameters,
    encoder forward + backward in PyTorch on a pseudo-user batch (16 sequences x 512 tokens), lambda-gradient
    reduction (A5), Adam on lambda (stack B of SURVEY.md section 3; `load_merging_module` + `DistillSequenceModule`'s
    optimiser set-up, sequence/module.py:94-100).  The two kernels of this package are timed inside the step and
    alone; the encoder is stock HF RoBERTa under bf16 autocast like the reference's Trainer (configs/base.py:41)."""

    name = "collab_cfg3"
    metric = "collaborative-merging steps/sec (lambda merge + encoder fwd/bwd + lambda-gradient + Adam)"
    unit = "steps/s"
    dtype = "f32 merge / lambda-gradient, bf16-autocast encoder"
    K = 8
    launches_per_step = 3   # merge_kernel, lg_partial_kernel, lg_finish kernel (the encoder's kernels are PyTorch's)
    e2e_steps_cap = 3

    def __init__(self, rank, world, device):
        super().__init__(rank, world, device)
        self.B, self.L = 16, 512
        self.shapes = synth.roberta_shapes()
        self.d = synth.total_numel(self.shapes)

    def config(self):
        return {"workload": "BASELINE config 3: collaborative merging step, K=8 BLaIR-base (RoBERTa-base, d=124,645,632), "
                            "layer-wise lambda (G=13), batch 16 x 512 tokens, Adam(lr 1e-3) on lambda",
                "K": self.K, "d": self.d, "batch": self.B, "seq_len": self.L,
                "l2": "4.5 GB of task vectors per merge / gradient pass exceed L2",
                "parallelism": "data-parallel replicas, one all-reduce of the G x K lambda-gradient per step (SURVEY.md 8(e))"}

    def setup(self):
        import torch.distributed as dist
        from transformers import RobertaConfig, RobertaModel
        from mergerec_b200.merger.enums import LearnType, MergeType
        from mergerec_b200.merger.weight_learning.module import load_merging_module

        class Wrapped(torch.nn.Module):      # the reference's BaseEncoderModel keeps the HF model under `.model`
            def __init__(self, hf):
                super().__init__()
                self.model = hf

            def forward(self, ids):
                return self.model(input_ids=ids).last_hidden_state[:, 0]   # CLS pooling (encoder/_base.py:32-39)

        torch.manual_seed(0)
        cfg = RobertaConfig(vocab_size=50265, max_position_embeddings=514, type_vocab_size=1, pad_token_id=1,
                            layer_norm_eps=1e-5, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
        model = Wrapped(RobertaModel(cfg, add_pooling_layer=True)).to(self.device)
        pre = {k: v.detach().clone() for k, v in model.state_dict().items()}
        g = torch.Generator(device=self.device).manual_seed(100 + self.rank)
        fts = [{k: (v + 1e-3 * torch.randn(v.shape, generator=g, device=self.device)) if v.is_floating_point() else v.clone()
                for k, v in pre.items()} for _ in range(self.K)]
        self.module = load_merging_module(MergeType.TASK_VECTOR, LearnType.LAYER_WISE, model, pre, fts, ignore_keys=set(),
                                          initial_per_weight=0.2, disable_softmax=True)
        del fts, pre
        self.opt = torch.optim.Adam(self.module.trainable_parameters(True, True, False), lr=1e-3)
        self.ids = torch.randint(3, 50000, (self.B, self.L), generator=g, device=self.device)
        self.group = dist.group.WORLD if self.world > 1 else None
        self.loss = None

    def step(self):
        import torch.distributed as dist
        self.opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            rep = self.module(self.ids)
        loss = rep.float().square().mean()
        loss.backward()
        if self.group is not None:
            for p in self.module.per_weights.parameters():
                dist.all_reduce(p.grad, op=dist.ReduceOp.AVG, group=self.group)
        self.opt.step()
        self.loss = loss.detach()

    def outputs(self):
        out = {"loss": _output(self.loss)}
        out.update({f"lambda.{k}": _output(v) for k, v in self.module.per_weights.items()})
        return out

    def units_per_step_all_ranks(self):
        return float(self.world)

    def setup_e2e(self):
        self.h_ids = _pinned(self.ids.cpu())
        self.h2d_bytes = self.h_ids.numel() * 8
        self.d2h_bytes = 4

    def step_e2e(self):
        self.ids.copy_(self.h_ids, non_blocking=True)
        self.step()
        float(self.loss)      # device -> host read of the step's loss

    def roofline(self, peaks):
        from bench import event_time_ms
        from mergerec_b200.merger.weight_learning.module._base import _lambda_grad
        m = self.module
        w = m._effective_weights().detach()
        ms_merge = event_time_ms(lambda: m._merge_flat(w), 10)
        _, seg_group, keys = m._blocks()
        grad = torch.randn(self.d, device=self.device)
        grads = [grad[o:o + n] for o, n in zip(m._layout.offsets, m._layout.sizes)]
        ms_grad = event_time_ms(lambda: _lambda_grad(grads, m._layout, m._task_rows(), seg_group, len(keys)), 10)
        # rank 0 only from here: with several ranks `step` holds an all-reduce, so time it only on one GPU
        ms_step = event_time_ms(self.step, 3) if self.world == 1 else None
        bytes_merge, bytes_grad = (self.K + 2) * self.d * 4, (self.K + 1) * self.d * 4
        ach = bytes_grad / GB / (ms_grad * 1e-3)
        return _with_traffic({"bound": "hbm", "kernel": "mr::lg_partial_kernel<8> (+ finish): lambda-gradient reduction (A5)",
                "achieved": ach, "peak": peaks["hbm_gbs"], "peak_source": peaks["source"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "traffic": None, "ms_per_launch": ms_grad,
                "algorithmic_bytes_per_launch": bytes_grad,
                "other_kernels": {"lambda merge forward (merge_kernel, A4)": {"ms": ms_merge, "GB/s": bytes_merge / GB / (ms_merge * 1e-3), "bytes": bytes_merge}},
                "step_ms": ms_step, "merge_plus_grad_share_of_step": None if ms_step is None else (ms_merge + ms_grad) / ms_step}, "lg_partial_kernel")

    def extra(self):
        return {"loss": None if self.loss is None else float(self.loss),
                "per_weights": {k: [round(x, 6) for x in v.tolist()] for k, v in list(self.module.per_weights.items())[:2]}}

    # -- CPU arm: the oracle port of the two merger kernels of the step (the encoder is PyTorch on both sides)
    def _cpu_time(self, reps):
        from oracle import oracle as orc
        rng = np.random.Generator(np.random.PCG64(7))
        d = self.d
        base = rng.standard_normal(d, dtype=np.float32) * np.float32(0.02)
        T = rng.standard_normal((self.K, d), dtype=np.float32) * np.float32(1e-3)
        sb, se, sg, keys = orc.segment_table(self.shapes, layer_wise=True)
        w = rng.uniform(0.1, 0.5, size=(len(keys), self.K)).astype(np.float32)
        grad = rng.standard_normal(d, dtype=np.float32)
        ts = []
        for _ in range(reps + 1):
            t0 = time.perf_counter()
            orc.lambda_merge(base, T, w, sb, se, sg)
            orc.lambda_grad(grad, T, len(keys), sb, se, sg)
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts[1:])), orc.max_threads()

    def cpu_baseline(self):
        t, cores = self._cpu_time(2)
        return {"value": 1.0 / t, "unit": self.unit, "cores": cores, "kind": "port",
                "sample": "the step's two merger passes only (lambda merge + lambda-gradient, full d, K=8), OpenMP C oracle "
                          "port; the encoder forward/backward is not included on the CPU side",
                "seconds_per_step": t}

    def reference_arm(self, steps, warmup):
        t, cores = self._cpu_time(max(1, steps))
        return {"value": 1.0 / t, "ms_per_step": t * 1e3, "cores": cores,
                "sample": "the step's two merger passes only (lambda merge + lambda-gradient, full d, K=8), OpenMP C oracle port"}


class TiesSharded(TiesCfg2):
    """SURVEY.md section 8(e), merger row: the TIES merge of BASELINE config 2 with the flat vector SHARDED over the
    ranks (d/G columns per GPU, 32-column aligned).  One step = global trim threshold (per-slice order statistic, then two
    sampled-bracket select `mr_ties_select_dist`: 4 all-reduces of 33 KB + 1 all-gather of 262 KB per rank, no host sync), TIES build of
    the local slice, task-wise lambda merge of the local slice.  Strong scaling: the whole job's algorithmic bytes
    ((2K+1) + (K+2)) * d * 4 divided by the slowest rank's time.  Results are bit-identical to the single-GPU merge
    (tests/test_sharded_merger_gpu.py)."""

    name = "ties_sharded"
    scaling = "strong"
    launches_per_step = 14  # init, 2 x sample pass, 5 x pick, full pass, 2 x cand_hist, compact, final, build, merge (+ NCCL's)

    def config(self):
        return {"workload": "TIES (density 0.2) of K=8 BLaIR-base models, flat vector sharded d/G per GPU; global trim via "
                            "all-reduced radix histograms; local build + task-wise lambda merge",
                "K": self.K, "d": self.d, "density": 0.2, "l2": "per-rank inputs (4.5 GB / G) exceed L2 for G <= 8",
                "parallelism": "flat dimension sharded d/G per GPU (strong scaling); per select 4 all-reduces of the K x 1024 "
                               "counters + 1 all-gather of the survivors; the same code path without collectives on 1 GPU"}

    def setup(self):
        import torch.distributed as dist
        from mergerec_b200.merger.layout import alloc_rows
        from mergerec_b200.merger.sharded import flat_shard_bounds
        g = torch.Generator(device=self.device).manual_seed(1234)    # same vectors on every rank, then keep the slice
        d, K = self.d, self.K
        lo, hi = flat_shard_bounds(d, self.world, self.rank)
        self.lo, self.hi = lo, hi
        base = torch.randn(d, generator=g, device=self.device) * 0.02
        self.models = []
        for _ in range(K):
            self.models.append((base + 1e-3 * torch.randn(d, generator=g, device=self.device))[lo:hi].clone())
        self.base = base[lo:hi].clone()
        del base
        self.group = dist.group.WORLD if self.world > 1 else None
        self.That = alloc_rows(K, hi - lo, self.device)
        self.Trows = list(self.That.unbind(0))
        self.w = torch.full((1, K), 0.3, dtype=torch.float32, device=self.device)
        self.out = torch.empty(hi - lo, dtype=torch.float32, device=self.device)

    def _select(self):
        """Stream-ordered device-side select (status checked after the timed loop, like the single-GPU step)."""
        from mergerec_b200.merger.sharded import sharded_select
        cut, self._status = sharded_select(self.base, self.models, int(0.2 * self.d), self.d, None, self.group, defer_status=True)
        return cut

    def _build(self, cut):
        from mergerec_b200 import _lib
        from mergerec_b200.merger.algorithms import ties as T
        T._build(self.base, self.models, cut, _lib.MR_TIES_VECTORS, out=self.That, ldo=max(self.That.stride(0), self.hi - self.lo))

    def _merge_only(self):
        from mergerec_b200 import _lib
        from mergerec_b200.merger.algorithms._common import merge_axpy
        merge_axpy(self.base, self.Trows, self.w, _lib.MR_ORDER_SUM_FIRST, False, out=self.out)

    def step(self):
        self._cut = self._select()
        self._build(self._cut)
        self._merge_only()

    def _e2e_kernels(self):
        self.step()

    def units_per_step_all_ranks(self):
        return self.bytes_per_step / GB      # strong scaling: one job, whatever the number of ranks

    def setup_e2e(self):
        # (every rank passes here once, after the timed loop) exact integer checksum of the merged vector's bit
        # patterns summed over the ranks: independent of the sharding because the sharded merge is bit-identical to
        # the single-GPU one -- compare the lines of different --gpus
        chk = self.out.view(torch.int32).to(torch.int64).sum().reshape(1)
        if self.group is not None:
            import torch.distributed as dist
            dist.all_reduce(chk, group=self.group)
        self._checksum = int(chk.item())
        n = self.hi - self.lo
        self.h_base = _pinned(self.base.cpu())
        self.h_models = [_pinned(m.cpu()) for m in self.models]
        self.h_out = torch.empty(n, dtype=torch.float32, pin_memory=True)
        self.h2d_bytes = (self.K + 1) * n * 4
        self.d2h_bytes = n * 4

    def roofline(self, peaks):
        from bench import event_time_ms
        n, K = self.hi - self.lo, self.K
        cut = self._cut                      # rank 0 only from here on: kernels, no collectives
        ms_select = event_time_ms(self._select, 5) if self.world == 1 else None
        ms_build = event_time_ms(lambda: self._build(cut), 10)
        ms_merge = event_time_ms(self._merge_only, 10)
        b_build, b_merge = (2 * K + 1) * n * 4, (K + 2) * n * 4
        ach = b_build / GB / (ms_build * 1e-3)
        return {"bound": "hbm", "kernel": "mr::ties_build_kernel<8, VECTORS, vec4> on this rank's slice",
                "achieved": ach, "peak": peaks["hbm_gbs"], "peak_source": peaks["source"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "traffic": None, "ms_per_launch": ms_build,
                "algorithmic_bytes_per_launch": b_build,
                "other_kernels": {
                    "device-side sharded select (mr_ties_select_dist: 2 sample passes + 1 full pass + finish; timed without "
                    "collectives, 1 GPU only)": {"ms": ms_select},
                    "lambda merge of the slice (merge_kernel)": {"ms": ms_merge, "GB/s": b_merge / GB / (ms_merge * 1e-3), "bytes": b_merge}}}

    def extra(self):
        return {"slice": [self.lo, self.hi], "merged_bits_checksum": self._checksum}


class PcbSharded(TiesSharded):
    """SURVEY.md section 8(e), merger row, for PCB merging (pcb.py:37-73): K = 8 BLaIR-base models, the flat vector
    SHARDED d/G over the ranks, the same seeded inputs as `ties_sharded`.  One step = `get_pcb_vectors_sharded` (two
    sharded magnitude selects for the 1 % / 99 % clamps, the phased quantile search `mr_pcb_vectors_dist` with all-reduced
    histograms, the build of the local slice; one host synchronisation for the status words) followed by the base-first
    merge of the slice.  Strong scaling: the whole job's algorithmic bytes divided by the slowest rank's time.  The merged
    slices are bit-identical to the single-GPU `merge_pcb` (tests/test_sharded_pcb_gpu.py); `merged_bits_checksum` is
    the same for every G."""

    name = "pcb_sharded"
    scaling = "strong"
    launches_per_step = 40  # 2 x 6-phase select, 7-phase search (incl. build), merge (+ NCCL's)

    def __init__(self, rank, world, device):
        super().__init__(rank, world, device)
        K, d = self.K, self.d
        # two clamp selects and the quantile search read base + K models once each, the build reads them and writes K
        # rows, the merge reads base + K rows and writes the result
        self.bytes_build = 3 * (K + 1) * d * 4 + (2 * K + 1) * d * 4
        self.bytes_merge = (K + 2) * d * 4
        self.bytes_per_step = self.bytes_build + self.bytes_merge

    def config(self):
        return {"workload": "PCB merge (density 0.2) of K=8 BLaIR-base models, flat vector sharded d/G per GPU; global "
                            "clamps and balancing-weight quantile via all-reduced radix histograms; local build + "
                            "base-first merge",
                "K": self.K, "d": self.d, "density": 0.2, "weights": 0.3,
                "l2": "per-rank inputs (4.5 GB / G) exceed L2 for G <= 8",
                "algorithmic_bytes": "3 x (K+1) d 4 (two clamp selects, quantile search) + (2K+1) d 4 (build) + (K+2) d 4 "
                                     "(merge)",
                "parallelism": "flat dimension sharded d/G per GPU (strong scaling); per step 2 x (4 all-reduces + 1 "
                               "all-gather) for the clamp selects, 6 all-reduces of the (2, K, 2048) histograms + 1 of "
                               "the row maxima for the quantile search, 1 all-reduce of the status words; the same code "
                               "path without collectives on 1 GPU"}

    def setup(self):
        super().setup()
        del self.That, self.Trows
        self.wl = [0.3] * self.K

    def _vectors(self):
        from mergerec_b200.merger.sharded import get_pcb_vectors_sharded
        self.vectors = get_pcb_vectors_sharded(self.base, self.models, 0.2, self.d, self.group)

    def _merge_only(self):
        from mergerec_b200 import _lib
        from mergerec_b200.merger.algorithms._common import merge_axpy, weights_tensor
        if self.hi > self.lo:
            merge_axpy(self.base, list(self.vectors.unbind(0)), weights_tensor(self.wl, self.device), _lib.MR_ORDER_BASE_FIRST,
                       False, out=self.out)

    def step(self):
        self._vectors()
        self._merge_only()

    def roofline(self, peaks):
        from bench import event_time_ms
        n, K = self.hi - self.lo, self.K
        ms_vec = event_time_ms(self._vectors, 3) if self.world == 1 else None     # collectives: every rank or none
        ms_merge = event_time_ms(self._merge_only, 10)
        b_merge = (K + 2) * n * 4
        ach = b_merge / GB / (ms_merge * 1e-3)
        return {"bound": "hbm", "kernel": "mr::merge_kernel (base-first PCB merge) on this rank's slice",
                "achieved": ach, "peak": peaks["hbm_gbs"], "peak_source": peaks["source"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "traffic": None, "ms_per_launch": ms_merge,
                "algorithmic_bytes_per_launch": b_merge,
                "other_kernels": {
                    "get_pcb_vectors_sharded (clamp selects + quantile search + build; timed without collectives, 1 GPU "
                    "only)": {"ms": ms_vec}}}

    # -- CPU arms: the unmodified reference `merge_pcb` (get_pcb_vectors + base-first sum) from baseline/_ref, and the
    #    numpy port of oracle/oracle.py beside it, both on a RoBERTa-shaped slice (12 layers, hidden 64, d = 3.85 M): at
    #    full size the reference sorts (K, 1.2e8) tensors three times per step.
    def _slice_inputs(self):
        shapes = synth.roberta_shapes(hidden=64, ffn=256)
        d = synth.total_numel(shapes)
        g = torch.Generator().manual_seed(7)
        base = torch.randn(d, generator=g) * 0.02
        models = [base + 1e-3 * torch.randn(d, generator=g) for _ in range(self.K)]
        return d, base, models

    def _port_step_fn(self):
        from oracle import oracle as orc
        d, base, models = self._slice_inputs()
        b, ms = base.numpy(), [m.numpy() for m in models]

        def step():
            orc.merge_pcb(b, ms, [0.3] * self.K, 0.2)
        nbytes = (4 * (self.K + 1) + self.K + (self.K + 2)) * d * 4
        return step, nbytes, (f"numpy port of get_pcb_vectors + merge_pcb (oracle/oracle.py) on a RoBERTa-shaped slice: 12 "
                              f"layers, hidden 64, d={d}, K={self.K}, density 0.2")

    def _reference_step_fn(self):
        ref = reference_package()
        if ref is None:
            return None
        from rec_retrieval.merger.algorithms.pcb import merge_pcb
        d, base, models = self._slice_inputs()

        def step():
            merge_pcb(base, models, [0.3] * self.K, density=0.2)
        nbytes = (4 * (self.K + 1) + self.K + (self.K + 2)) * d * 4
        return step, nbytes, (f"UNMODIFIED reference merge_pcb (get_pcb_vectors + base-first sum) on a RoBERTa-shaped slice: "
                              f"12 layers, hidden 64, d={d}, K={self.K}, density 0.2")


class DistillStep(Workload):
    """The distillation half of a collaborative-merging step (SURVEY.md section 8(f) rank 1; reference:
    module/distiller/sequence/module.py:59-76 + loss_fn.py KD loss): catalogue logits of 16 pseudo-user representations
    against their domains' item tables (8 domains x 25,000 items, E = 768 -- the per-domain share of BASELINE config 4's
    200K-item union catalogue), KD loss against device-resident teacher logits, gradient w.r.t. the representations.
    Algorithmic bytes per step: every used item table once in the forward and once in the backward pass."""

    name = "distill_step"
    metric = "distillation samples/sec (catalogue logits + KD loss + representation gradient)"
    unit = "samples/s"
    dtype = "f32"
    launches_per_step = 4     # ds_logits, ds_loss, ds_grad, ds_grad_finish
    D, N, E, B, NSEQ = 8, 25000, 768, 16, 512

    def config(self):
        return {"workload": "distillation step: 16 samples over 8 domains x 25,000 items, E=768, KD loss (T=2), "
                            "teacher logits device-resident (512 sequences per domain)",
                "B": self.B, "domains": self.D, "items_per_domain": self.N, "E": self.E,
                "l2": "item tables (614 MB) exceed L2",
                "parallelism": "independent replicas (no collective on this path)"}

    def setup(self):
        from mergerec_b200.module.distiller import TeacherScores
        from mergerec_b200.module.recommender.loss_fn import DistillKDLoss
        g = torch.Generator(device=self.device).manual_seed(77 + self.rank)
        mk = lambda *shape: torch.randn(*shape, generator=g, device=self.device)
        t_items = [mk(self.N, self.E) for _ in range(self.D)]
        t_seqs = [mk(self.NSEQ, self.E) for _ in range(self.D)]
        self.teacher = TeacherScores(t_items, t_seqs)
        self.tables = [torch.nn.functional.normalize(t, dim=-1) + 0.02 * mk(self.N, self.E) for t in t_items]
        self.dom = [b % self.D for b in range(self.B)]
        self.seq_ids = [int(x) for x in torch.randint(0, self.NSEQ, (self.B,), generator=g, device=self.device).tolist()]
        self.rep = torch.nn.functional.normalize(torch.stack([t_seqs[d][s] for d, s in zip(self.dom, self.seq_ids)]) + 0.3 * mk(self.B, self.E), dim=-1)
        self.rep.requires_grad_(True)
        self.spec = DistillKDLoss(2.0).spec
        _, self.ptrs = self.teacher.rows(self.dom, self.seq_ids)
        self.bytes_tables = self.D * self.N * self.E * 4
        self.loss = None
        self._try_capture()

    def _eager_step(self):
        from mergerec_b200.module.distiller.sequence.module import fused_distill_losses
        self.rep.grad = None
        loss = fused_distill_losses(self.rep, self.tables, self.dom, self.ptrs, self.spec).mean()
        loss.backward()
        self.loss = loss.detach()

    def _try_capture(self):
        """The step is launch-bound (about ten launches for ~0.23 ms of GPU work): capture forward + backward in one CUDA
        graph and replay it.  Every entry point of the C ABI is stream-ordered and takes its small tables by value, so
        the capture needs nothing special; if it fails for any reason the eager step stays."""
        self.graph = None
        if os.environ.get("MR_BENCH_NO_GRAPH"):
            return
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    self._eager_step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            self.rep.grad = None
            with torch.cuda.graph(g):
                self._eager_step()
            g.replay()
            torch.cuda.synchronize()
            self.graph = g
        except Exception as e:  # noqa: BLE001 -- report, keep the eager path
            print(f"[distill_step] CUDA graph capture unavailable ({type(e).__name__}: {e}); eager launches", file=__import__("sys").stderr)
            self.graph = None
            torch.cuda.synchronize()

    def step(self):
        if getattr(self, "graph", None) is not None:
            self.graph.replay()
        else:
            self._eager_step()

    def outputs(self):
        return {"loss": _output(self.loss), "rep_grad": _output(self.rep.grad)}

    def units_per_step_all_ranks(self):
        return float(self.B * self.world)

    def setup_e2e(self):
        self.h_rep = _pinned(self.rep.detach().cpu())
        self.h_grad = torch.empty((self.B, self.E), dtype=torch.float32, pin_memory=True)
        self.h2d_bytes = self.B * self.E * 4
        self.d2h_bytes = self.B * self.E * 4 + 4

    def step_e2e(self):
        with torch.no_grad():
            self.rep.copy_(self.h_rep, non_blocking=True)
        if getattr(self, "graph", None) is None:
            _, self.ptrs = self.teacher.rows(self.dom, self.seq_ids)
        self.step()
        self.h_grad.copy_(self.rep.grad, non_blocking=True)
        float(self.loss)

    def roofline(self, peaks):
        from bench import event_time_ms
        from mergerec_b200.module.distiller.sequence.module import distill_logits
        rep = self.rep.detach()
        out = distill_logits(rep, self.tables, self.dom)
        ms = event_time_ms(lambda: distill_logits(rep, self.tables, self.dom, out=out), 20)
        ms_step = event_time_ms(self.step, 10)
        ach = self.bytes_tables / GB / (ms * 1e-3)
        return _with_traffic({"bound": "hbm", "kernel": "mr::ds_logits_kernel<6, 2> (catalogue logits, every item table read once)",
                "achieved": ach, "peak": peaks["hbm_gbs"], "peak_source": peaks["source"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "traffic": None, "ms_per_launch": ms,
                "algorithmic_bytes_per_launch": self.bytes_tables, "step_ms": ms_step,
                "step_GB/s (tables read twice)": 2 * self.bytes_tables / GB / (ms_step * 1e-3)}, "ds_logits_kernel")

    def extra(self):
        return {"loss": None if self.loss is None else float(self.loss), "cuda_graph": getattr(self, "graph", None) is not None}

    def _cpu_time(self, reps):
        from oracle import oracle as orc
        rng = np.random.Generator(np.random.PCG64(7))
        tables = [rng.standard_normal((self.N, self.E), dtype=np.float32) * np.float32(0.05) for _ in range(self.D)]
        rep = rng.standard_normal((self.B, self.E), dtype=np.float32)
        trows = [rng.standard_normal(self.N, dtype=np.float32) for _ in range(self.B)]
        ts = []
        for _ in range(reps + 1):
            t0 = time.perf_counter()
            orc.distill_step(rep, tables, self.dom if hasattr(self, "dom") else [b % self.D for b in range(self.B)], trows, "KD", temperature=2.0)
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts[1:])), os.cpu_count() or 1

    def cpu_baseline(self):
        t, cores = self._cpu_time(2)
        return {"value": self.B / t, "unit": self.unit, "cores": cores, "kind": "port",
                "sample": "the full step (16 samples, 8 x 25,000 x 768 tables), numpy fp64 oracle port (BLAS threads)", "seconds_per_step": t}

    def reference_arm(self, steps, warmup):
        t, cores = self._cpu_time(max(1, steps))
        return {"value": self.B / t, "ms_per_step": t * 1e3, "cores": cores,
                "sample": "the full step (16 samples, 8 x 25,000 x 768 tables), numpy fp64 oracle port"}


class TaskArithCfg1(LambdaMergeK8):
    """Merger half of BASELINE config 1: task-arithmetic merge of K = 3 BLaIR-base domain models, lambda = 0.3
    (`ModelMerger.merge("task_vector", 0.3)`, merger.py:71-74 -> task_vector.py:13-34).  Algorithmic bytes per step:
    (K+2) * d * 4.  The end-to-end arm is the public API itself: host state_dicts -> `ModelMerger` (flatten into HBM) ->
    merge -> merged flat vector back to the host."""

    name = "task_arith_cfg1"
    K = 3

    def config(self):
        return {"workload": "BASELINE config 1 (merger half): task-arithmetic merge of K=3 BLaIR-base (RoBERTa-base, "
                            "d=124,645,632, P=199) domain models, lambda=0.3",
                "K": self.K, "d": self.d, "l2": "inputs (2 GB) exceed L2, no flush needed",
                "parallelism": "single GPU"}

    def setup(self):
        g = torch.Generator(device=self.device).manual_seed(1234)
        d, K = self.d, self.K
        self.base = torch.randn(d, generator=g, device=self.device) * 0.02
        self.models = [self.base + 1e-3 * torch.randn(d, generator=g, device=self.device) for _ in range(K)]
        self.w = torch.full((1, K), 0.3, dtype=torch.float32, device=self.device)
        self.out = torch.empty(d, dtype=torch.float32, device=self.device)

    def step(self):
        from mergerec_b200 import _lib
        from mergerec_b200.merger.algorithms._common import merge_axpy
        merge_axpy(self.base, self.models, self.w, _lib.MR_ORDER_BASE_FIRST, True, out=self.out)

    def setup_e2e(self):
        from mergerec_b200.merger.layout import FlatLayout
        layout = FlatLayout.from_shape_dict(self.shapes)
        self.h_flat = [_pinned(t.cpu()) for t in [self.base] + self.models]
        self.h_dicts = [layout.views(f) for f in self.h_flat]          # host state_dicts (views of pinned flat buffers)
        self.h_out = torch.empty(self.d, dtype=torch.float32, pin_memory=True)
        self.h2d_bytes = (self.K + 1) * self.d * 4
        self.d2h_bytes = self.d * 4
        del self.base, self.models
        torch.cuda.empty_cache()

    def step_e2e(self):
        from mergerec_b200.merger import ModelMerger
        merger = ModelMerger(self.h_dicts[1:], self.h_dicts[0], align_key_order=False)
        merged = merger.merge("task_vector", 0.3)
        first = next(iter(merged.values()))
        flat = first.reshape(-1)
        # the merged state_dict's tensors are views of one flat device vector in layout order: copy it back whole
        self.h_out.copy_(torch.as_strided(flat, (self.d,), (1,), first.storage_offset()), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def teardown_e2e(self):
        g = torch.Generator(device=self.device).manual_seed(1234)
        d, K = self.d, self.K
        self.base = torch.randn(d, generator=g, device=self.device) * 0.02
        self.models = [self.base + 1e-3 * torch.randn(d, generator=g, device=self.device) for _ in range(K)]
        del self.h_flat, self.h_dicts

    def roofline(self, peaks):
        from bench import event_time_ms
        ms = event_time_ms(self.step, 20)
        achieved = self.bytes_per_step / GB / (ms * 1e-3)
        return _with_traffic({"bound": "hbm", "kernel": "mr::merge_kernel<3, BASE_FIRST, src_is_model, vec4>", "achieved": achieved,
                "peak": peaks["hbm_gbs"], "peak_source": peaks["source"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": None, "ms_per_launch": ms,
                "algorithmic_bytes_per_launch": self.bytes_per_step}, "merge_kernel")

    # -- CPU arms at FULL size: the unmodified ModelMerger.merge("task_vector", 0.3) (reference) / oracle port
    def _host_models(self):
        base, models = synth.make_state_dicts(self.shapes, self.K, seed=0, sigma=1e-3)
        return base, models

    def _reference_step_fn(self):
        if reference_package() is None:
            return None
        from rec_retrieval.merger import ModelMerger as RefMerger
        base, models = self._host_models()
        t0 = time.perf_counter()
        merger = RefMerger([{k: torch.from_numpy(v) for k, v in m.items()} for m in models],
                           {k: torch.from_numpy(v) for k, v in base.items()})
        t_flat = time.perf_counter() - t0
        del base, models
        return (lambda: merger.merge("task_vector", 0.3)), self.bytes_per_step, (
            f"UNMODIFIED reference ModelMerger.merge('task_vector', 0.3) at the full size (K={self.K}, d={self.d}); the "
            f"constructor's flatten_model x{self.K + 1} took {t_flat:.2f} s and is not in the step")

    def _port_step_fn(self):
        from oracle import oracle as orc
        rng = np.random.Generator(np.random.PCG64(7))
        base = rng.standard_normal(self.d, dtype=np.float32) * np.float32(0.02)
        models = [base + np.float32(1e-3) * rng.standard_normal(self.d, dtype=np.float32) for _ in range(self.K)]
        return (lambda: orc.merge_task_vector(base, models, [0.3] * self.K)), self.bytes_per_step, (
            f"full size (K={self.K}, d={self.d}) merge_task_vector, OpenMP C oracle port")

    cpu_baseline = TiesCfg2.cpu_baseline
    reference_arm = TiesCfg2.reference_arm


class MergeCfg4(TiesCfg2):
    """Merger half of BASELINE config 4: K = 8 Recformer-large (Longformer-large, d = 433,610,754, P = 535) domain models.
    One step = task-arithmetic merge from the models (A1) + `get_ties_vectors(density 0.2)` (A6-A8) + task-wise lambda
    merge of the TIES vectors (A3).  Algorithmic bytes per step: (K+2)*d*4 + (2K+1)*d*4 + (K+2)*d*4 = 64.2 GB."""

    name = "merge_cfg4"
    launches_per_step = 13
    e2e_steps_cap = 2

    def __init__(self, rank, world, device):
        Workload.__init__(self, rank, world, device)
        self.shapes = synth.recformer_shapes()
        self.d = synth.total_numel(self.shapes)
        self.bytes_arith = (self.K + 2) * self.d * 4
        self.bytes_build = (2 * self.K + 1) * self.d * 4
        self.bytes_merge = (self.K + 2) * self.d * 4
        self.bytes_per_step = self.bytes_arith + self.bytes_build + self.bytes_merge

    def config(self):
        return {"workload": "BASELINE config 4 (merger half): K=8 Recformer-large (Longformer-large, d=433,610,754, P=535; flat "
                            "offsets after position_ids are 2 mod 4): task-arithmetic merge + TIES vectors (density 0.2, global "
                            "trim, election, disjoint mean) + task-wise lambda merge",
                "K": self.K, "d": self.d, "density": 0.2, "l2": "inputs (15.6 GB) exceed L2, no flush needed",
                "select_status": "checked on the host after the timed loop (stream-ordered step)",
                "parallelism": "single GPU"}

    def setup(self):
        from mergerec_b200.merger.layout import alloc_rows
        g = torch.Generator(device=self.device).manual_seed(4321)
        d, K = self.d, self.K
        self.base = torch.randn(d, generator=g, device=self.device) * 0.02
        self.models = []
        for _ in range(K):
            m = torch.randn(d, generator=g, device=self.device)
            m.mul_(1e-3).add_(self.base)
            self.models.append(m)
        self.w_arith = torch.full((1, K), 0.3, dtype=torch.float32, device=self.device)
        rng = np.random.Generator(np.random.PCG64(5))
        self.w = torch.from_numpy(rng.uniform(0.1, 0.5, size=(1, K)).astype(np.float32)).to(self.device)
        self.out = torch.empty(d, dtype=torch.float32, device=self.device)
        self.out_arith = torch.empty(d, dtype=torch.float32, device=self.device)
        self.That = alloc_rows(K, d, self.device)
        self.Trows = list(self.That.unbind(0))
        self.seg_end = self.seg_group = None
        self._status = None
        self.graph = None

    def _arith(self):
        from mergerec_b200 import _lib
        from mergerec_b200.merger.algorithms._common import merge_axpy
        merge_axpy(self.base, self.models, self.w_arith, _lib.MR_ORDER_BASE_FIRST, True, out=self.out_arith)

    def _eager_step(self, defer=True):
        self._arith()
        TiesCfg2._eager_step(self, defer)

    def step(self):
        self._eager_step()

    def outputs(self):
        return {"task_arithmetic": _output(self.out_arith), "merged": _output(self.out)}

    def step_fused(self):
        from mergerec_b200.merger.algorithms import ties as T
        T.merge_ties_lambda(self.base, self.models, 0.2, self.w, out=self.out)

    def setup_e2e(self):
        self.h_base = _pinned(self.base.cpu())
        self.h_models = [_pinned(m.cpu()) for m in self.models]
        self.h_out = torch.empty(self.d, dtype=torch.float32, pin_memory=True)
        self.h_out_arith = torch.empty(self.d, dtype=torch.float32, pin_memory=True)
        self.h2d_bytes = (self.K + 1) * self.d * 4
        self.d2h_bytes = 2 * self.d * 4

    def step_e2e(self):
        self.base.copy_(self.h_base, non_blocking=True)
        for m, h in zip(self.models, self.h_models):
            m.copy_(h, non_blocking=True)
        self._eager_step(defer=False)
        self.h_out_arith.copy_(self.out_arith, non_blocking=True)
        self.h_out.copy_(self.out, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def teardown_e2e(self):
        del self.h_base, self.h_models, self.h_out, self.h_out_arith

    def roofline(self, peaks):
        from bench import event_time_ms
        from mergerec_b200 import _lib
        from mergerec_b200.merger.algorithms import ties as T
        cut = T.ties_select(self.base, self.models, 0.2)
        K, d = self.K, self.d
        ms_build = event_time_ms(lambda: T._build(self.base, self.models, cut, _lib.MR_TIES_VECTORS, out=self.That, ldo=self.That.stride(0)), 5)
        ms_select = event_time_ms(lambda: T.select_kth_largest(self.base, self.models, int(0.2 * d), None, defer_status=True), 5)
        ms_merge = event_time_ms(self._merge_only, 5)
        ms_arith = event_time_ms(self._arith, 5)
        ms_fused = event_time_ms(self.step_fused, 3)
        ach = self.bytes_build / GB / (ms_build * 1e-3)
        sel_bytes = (K + 1) * d * 4
        return {"bound": "hbm", "kernel": "mr::ties_build_kernel<8, VECTORS, vec4> at d=433,610,754 (get_ties_vectors build pass)",
                "achieved": ach, "peak": peaks["hbm_gbs"], "peak_source": peaks["source"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "traffic": None, "ms_per_launch": ms_build,
                "algorithmic_bytes_per_launch": self.bytes_build,
                "other_kernels": {
                    "task-arithmetic merge from models (merge_kernel, A1)": {"ms": ms_arith, "GB/s": self.bytes_arith / GB / (ms_arith * 1e-3), "bytes": self.bytes_arith},
                    "ties_select (sample + 1 full pass + finish)": {"ms": ms_select, "GB/s": sel_bytes / GB / (ms_select * 1e-3), "bytes": sel_bytes},
                    "task-wise lambda merge of That (merge_kernel, A3)": {"ms": ms_merge, "GB/s": self.bytes_merge / GB / (ms_merge * 1e-3), "bytes": self.bytes_merge},
                    "fused TIES + lambda merge in one pass, That never materialised (merge_ties_lambda)": {"ms": ms_fused, "GB/s": self.bytes_merge / GB / (ms_fused * 1e-3), "bytes": self.bytes_merge},
                }}

    def extra(self):
        return {}

    # -- CPU arms on bounded samples (the full size needs ~45 GB of host temporaries and minutes per step on the CPU)
    def _port_step_fn(self):
        from oracle import oracle as orc
        frac = 8
        d = self.d // frac
        rng = np.random.Generator(np.random.PCG64(7))
        base = rng.standard_normal(d, dtype=np.float32) * np.float32(0.02)
        models = [base + np.float32(1e-3) * rng.standard_normal(d, dtype=np.float32) for _ in range(self.K)]
        w = rng.uniform(0.1, 0.5, size=(1, self.K)).astype(np.float32)

        def step():
            orc.merge_task_vector(base, models, [0.3] * self.K)
            That = orc.ties_vectors(base, models, 0.2)
            orc.lambda_merge(base, That, w)
        nbytes = ((self.K + 2) + (2 * self.K + 1) + (self.K + 2)) * d * 4
        return step, nbytes, (f"a flat prefix of d/{frac} = {d} elements, K={self.K}: merge_task_vector + ties_vectors + task-wise "
                              "lambda merge, OpenMP C oracle port")

    def _reference_step_fn(self):
        if reference_package() is None:
            return None
        from rec_retrieval.merger.algorithms.task_vector import merge_task_vector
        from rec_retrieval.merger.algorithms.ties import get_ties_vectors
        from rec_retrieval.merger.weight_learning.module.task_wise import TaskVectorMergingModuleTaskWise
        shapes = synth.recformer_shapes(hidden=64, ffn=256)
        d = synth.total_numel(shapes)
        g = torch.Generator().manual_seed(7)
        base = torch.randn(d, generator=g) * 0.02
        models = [base + 1e-3 * torch.randn(d, generator=g) for _ in range(self.K)]
        shape_dict = {k: torch.Size(v) for k, v in shapes.items()}

        class _NoModel(torch.nn.Module):
            def forward(self, x):
                return x

        def step():
            merge_task_vector(base, models, [0.3] * self.K)
            That = get_ties_vectors(base, models, 0.2)
            mod = TaskVectorMergingModuleTaskWise(base, That, _NoModel(), shape_dict, disable_softmax=True)
            with torch.no_grad():
                mod._merge_task_vectors()
        nbytes = ((self.K + 2) + (2 * self.K + 1) + (self.K + 2)) * d * 4
        return step, nbytes, ("UNMODIFIED reference (merge_task_vector + get_ties_vectors + TaskVectorMergingModuleTaskWise."
                              f"_merge_task_vectors) on a Recformer-shaped slice: 24 layers, hidden 64, P=535, d={d}, K={self.K}")


class EvalCfg1(EvalCatalog):
    """BASELINE config 1: Recall@10 / NDCG@10 of 256 query sequences against a 20,000-item catalog, E = 768 (the
    reference's own CPU-runnable case), with the K = 3 task-arithmetic merge carried as the `merger` object.  The CPU arms
    run at the FULL size of the configuration."""

    name = "cfg1"
    label = "BASELINE config 1"
    sizes = dict(Q=256, N=20_000, E=768, K=10)
    ks_low = 10
    cpu_sample = dict(Q=256)
    accuracy_rows = 256
    e2e_steps_cap = 10

    def companion(self):
        return TaskArithCfg1 if self.world == 1 else None


class EvalCfg4(EvalCatalog):
    """BASELINE config 4: evaluation over the 8-domain union catalog -- 200,000 items, E = 1024 (Recformer-large),
    Q = 32,768 query sequences, top-50 (the reference default max(ks), configs/base.py:46-48) -- with the Recformer-large
    K = 8 merge carried as the `merger` object."""

    name = "cfg4"
    label = "BASELINE config 4"
    sizes = dict(Q=32768, N=200_000, E=1024, K=50)
    ks_low = 10
    cpu_sample = dict(Q=512)
    accuracy_rows = 2048

    def companion(self):
        return MergeCfg4 if self.world == 1 else None


WORKLOADS = {LambdaMergeK8.name: LambdaMergeK8, TiesCfg2.name: TiesCfg2, EvalCatalog.name: EvalCatalog,
             CollabStepCfg3.name: CollabStepCfg3, DistillStep.name: DistillStep, TiesSharded.name: TiesSharded,
             PcbSharded.name: PcbSharded,
             TaskArithCfg1.name: TaskArithCfg1, MergeCfg4.name: MergeCfg4, EvalCfg1.name: EvalCfg1, EvalCfg4.name: EvalCfg4}
DEFAULT_WORKLOAD = EvalCatalog.name
