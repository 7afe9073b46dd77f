"""GPU: the sharded merger with the real kernels.  `mr_ties_mag_hist` against numpy; world size 1 in-process; and two
processes sharing one GPU (gloo for the small collectives -- NCCL refuses two ranks on one device) must reproduce the
single-GPU `get_ties_vectors` / `merge_ties` / `merge_task_vector` / `ModelMerger.merge` results bit for bit."""
import multiprocessing as mp
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist

from mergerec_b200 import synth
from mergerec_b200.merger import ModelMerger
from mergerec_b200.merger.algorithms import get_ties_vectors, merge_linear, merge_task_vector, merge_ties
from mergerec_b200.merger.sharded import (CudaKernels, ShardedModelMerger, flat_shard_bounds, gather_flat,
                                          get_ties_vectors_sharded, merge_linear_sharded, merge_task_vector_sharded,
                                          merge_ties_sharded)
from sharded_helpers import OracleKernels
from test_sharded_merger_host import CASES, _case_inputs, _free_port

pytestmark = pytest.mark.gpu


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("K,d,w", [(3, 4165, False), (8, 100003, True), (16, 777, True)])
def test_mag_hist_matches_numpy(K, d, w):
    base, models = synth.make_flat(d, K, seed=5, quantize=2.5e-4)
    wt = torch.linspace(0.1, 0.9, K) if w else None
    rng = np.random.default_rng(1)
    med, _ = OracleKernels.kth_largest_bits(torch.from_numpy(base), [torch.from_numpy(m) for m in models], d // 5, wt)
    for lo, shift in ((torch.zeros(K, dtype=torch.int64), torch.full((K,), 20)),                 # full range
                      ((med - (1 << 17)).clamp(min=0), torch.full((K,), 7)),                      # the usual first window
                      (med, torch.zeros(K, dtype=torch.int64)),                                   # single bit patterns
                      (torch.from_numpy(rng.integers(0, 2 ** 30, K)), torch.from_numpy(rng.integers(0, 21, K)))):
        got_h = torch.zeros((K, 2048), dtype=torch.int64, device="cuda")
        got_a = torch.zeros(K, dtype=torch.int64, device="cuda")
        CudaKernels.mag_hist(dev(base), [dev(m) for m in models], None if wt is None else wt.cuda(),
                             lo.cuda().to(torch.int32), shift.cuda().to(torch.int32), got_h, got_a)
        want_h, want_a = torch.zeros((K, 2048), dtype=torch.int64), torch.zeros(K, dtype=torch.int64)
        OracleKernels.mag_hist(torch.from_numpy(base), [torch.from_numpy(m) for m in models], wt, lo, shift, want_h, want_a)
        assert torch.equal(got_h.cpu(), want_h) and torch.equal(got_a.cpu(), want_a)
    unaligned = [dev(np.concatenate([[0.0], m]).astype(np.float32))[1:] for m in models]         # scalar path
    got_h.zero_(); got_a.zero_()
    CudaKernels.mag_hist(dev(base), unaligned, None if wt is None else wt.cuda(), lo.cuda().to(torch.int32),
                         shift.cuda().to(torch.int32), got_h, got_a)
    assert torch.equal(got_h.cpu(), want_h) and torch.equal(got_a.cpu(), want_a)


def _compare(case, group, world, rank):
    """Names of the checks that failed (empty list = all bit-identical)."""
    base, models = _case_inputs(case)
    d = case["d"]
    lo, hi = flat_shard_bounds(d, world, rank)
    fb, fm = dev(base), [dev(m) for m in models]
    bl, ml = fb[lo:hi].clone(), [m[lo:hi].clone() for m in fm]
    bad = []
    if not torch.equal(get_ties_vectors_sharded(bl, ml, case["density"], d, group)[:, :hi - lo],
                       get_ties_vectors(fb, fm, case["density"])[:, lo:hi]):
        bad.append("ties_vectors")
    if not torch.equal(gather_flat(merge_ties_sharded(bl, ml, case["weights"], case["density"], d, group), d, group),
                       merge_ties(fb, fm, case["weights"], case["density"])):
        bad.append("merge_ties")
    if not torch.equal(gather_flat(merge_task_vector_sharded(bl, ml, case["weights"]), d, group),
                       merge_task_vector(fb, fm, case["weights"])):
        bad.append("task_vector")
    if not torch.equal(gather_flat(merge_linear_sharded(ml, case["weights"]), d, group),
                       merge_linear(models=fm, weights=case["weights"])):
        bad.append("linear")
    return [f"d={d},K={case['K']}:{b}" for b in bad]


def test_world1_matches_single_gpu_paths():
    for case in CASES:
        assert _compare(case, None, 1, 0) == [], case


def _model_merger_check(group):
    shapes = synth.tiny_shapes(recformer=True)
    base, models = synth.make_state_dicts(shapes, 5, seed=22, sigma=1e-2)
    to_t = lambda sd: {k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}
    base, models = to_t(base), [to_t(m) for m in models]
    ref = ModelMerger(models, base)
    sh = ShardedModelMerger(models, base, group=group)
    bad = []
    for mt, w, kw in (("task_vector", 0.3, {}), ("linear", [0.1, 0.2, 0.3, 0.2, 0.2], {}), ("ties", 0.4, dict(density=0.2))):
        a, b = ref.merge(mt, w, **kw), sh.merge(mt, w, **kw)
        if not (list(a.keys()) == list(b.keys()) and all(torch.equal(a[k], b[k]) for k in a)):
            bad.append(f"ModelMerger:{mt}")
    return bad


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.cuda.set_device(0)
        bad = [b for case in CASES for b in _compare(case, dist.group.WORLD, world, rank)]
        bad += _model_merger_check(dist.group.WORLD)
        q.put((rank, bad))
    except Exception as e:  # noqa: BLE001
        import traceback
        q.put((rank, repr(e) + traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def test_two_ranks_on_one_gpu_bit_identical():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert sorted(results) == [(0, []), (1, [])]


def test_full_size_world1_select_agrees_with_the_bracket_select():
    """BLaIR-base, K = 8: the radix-histogram select (sharded path, world 1) and the sampled-bracket select (single-GPU
    path) must produce identical TIES vectors."""
    d, K = synth.total_numel(synth.roberta_shapes()), 8
    g = torch.Generator(device="cuda").manual_seed(11)
    base = torch.randn(d, generator=g, device="cuda") * 0.02
    models = [base + 1e-3 * torch.randn(d, generator=g, device="cuda") for _ in range(K)]
    a = get_ties_vectors_sharded(base, models, 0.2, d, None)
    b = get_ties_vectors(base, models, 0.2)
    assert torch.equal(a[:, :d], b[:, :d])


# ------------------------------------------------------------------------------------------ device-side sharded select
def _emulated_dist_select(base, models, k_cnt, world, w=None):
    """Run `world` DistSelect instances (one per emulated rank) on this GPU, playing the collectives by hand: sum the
    counters views after phases 0-3, concatenate the survivors regions after phase 4."""
    from mergerec_b200.merger.sharded import DistSelect
    d = base.numel()
    sels = []
    for r in range(world):
        lo, hi = flat_shard_bounds(d, world, r)
        sels.append(DistSelect(base[lo:hi].clone(), [m[lo:hi].clone() for m in models], k_cnt, d, lo, w))
    gathered = None
    for phase in range(DistSelect.PHASES):
        for s in sels:
            s.run(phase, gathered, world)
        if phase < 4:
            total = torch.stack([s.counters for s in sels]).sum(0, dtype=torch.int32)
            for s in sels:
                s.counters.copy_(total)
        elif phase == 4:
            gathered = torch.cat([s.survivors for s in sels])
    return sels


@pytest.mark.parametrize("K,d,world,quantize,weighted", [(3, 200_003, 2, 0.0, False), (8, 1_000_003, 4, 0.0, False),
                                                         (5, 300_031, 3, 2.5e-4, True), (8, 524_288, 8, 1e-5, False),
                                                         (2, 4099, 5, 0.0, False), (16, 100_001, 2, 0.0, True)])
def test_dist_select_emulated_ranks_equal_single_gpu(K, d, world, quantize, weighted):
    """The phased device-side select over `world` slices (collectives played by hand) gives the single-GPU cut keys, and
    the per-rank local cuts rebuild exactly the single-GPU TIES vectors / merge_ties on every slice."""
    from mergerec_b200 import _lib
    from mergerec_b200.merger.algorithms.ties import _build, select_kth_largest
    from mergerec_b200.merger.layout import alloc_rows
    base, models = synth.make_flat(d, K, seed=40 + K, quantize=quantize)
    fb, fm = dev(base), [dev(m) for m in models]
    w = torch.linspace(0.2, 1.1, K).cuda() if weighted else None
    k_cnt = int(0.2 * d)
    want_cut = select_kth_largest(fb, fm, k_cnt, w)
    sels = _emulated_dist_select(fb, fm, k_cnt, world, w)
    statuses = [s.status.cpu().tolist() for s in sels]
    assert all(st == statuses[0] for st in statuses), f"ranks disagree on the verdict: {statuses}"
    ok = torch.tensor(statuses[0]) == 1
    assert set(statuses[0]) <= {1, -1, -2, -3, -4, -5}, statuses[0]
    for r, s in enumerate(sels):
        assert torch.equal(s.cut_global.cpu()[ok], want_cut.cpu()[ok]), f"rank {r}: global cut, status 1"
    if statuses[0] != [1] * K:
        # thousands of equal magnitudes AT the cut (quantised inputs): two 1024-way refinements cannot separate them;
        # every rank reports it and `sharded_select` takes the exact path, which must still give the exact cut
        assert quantize > 0, f"fast select failed on a tie-free input: {statuses[0]}"
        from mergerec_b200.merger.sharded import sharded_select
        assert torch.equal(sharded_select(fb, fm, k_cnt, d, w), want_cut)
        return
    mode = _lib.MR_TIES_TRIMSUM if weighted else _lib.MR_TIES_VECTORS
    full = torch.empty(d, device="cuda") if weighted else alloc_rows(K, d, "cuda")
    _build(fb, fm, want_cut, mode, w=w, out=full, ldo=0 if weighted else max(full.stride(0), d))
    for r, s in enumerate(sels):
        lo, hi = flat_shard_bounds(d, world, r)
        if hi == lo:
            continue
        part = torch.empty(hi - lo, device="cuda") if weighted else alloc_rows(K, hi - lo, "cuda")
        _build(s.base, s.rows, s.cut, mode, w=w, out=part, ldo=0 if weighted else max(part.stride(0), hi - lo))
        if weighted:
            assert torch.equal(part.view(torch.int32), full[lo:hi].view(torch.int32)), f"rank {r}: merge_ties slice"
        else:
            assert torch.equal(part[:, :hi - lo].view(torch.int32), full[:, lo:hi].view(torch.int32)), f"rank {r}: TIES vectors slice"


def test_dist_select_world1_and_fallback():
    """group=None goes through the same phased kernels (no collective); an input the sampled bracket cannot resolve
    (every magnitude equal) falls back to the exact windowed search and still returns the exact cut."""
    from mergerec_b200.merger.algorithms.ties import select_kth_largest
    from mergerec_b200.merger.sharded import sharded_select
    base, models = synth.make_flat(150_001, 4, seed=9)
    fb, fm = dev(base), [dev(m) for m in models]
    k = int(0.2 * 150_001)
    cut, status = sharded_select(fb, fm, k, 150_001, defer_status=True)
    assert status.cpu().tolist() == [1] * 4 and torch.equal(cut, select_kth_largest(fb, fm, k))
    zb = torch.zeros(100_000, device="cuda")
    zm = [torch.full((100_000,), 0.5, device="cuda"), torch.full((100_000,), -0.5, device="cuda")]
    assert torch.equal(sharded_select(zb, zm, 20_000, 100_000), select_kth_largest(zb, zm, 20_000))
