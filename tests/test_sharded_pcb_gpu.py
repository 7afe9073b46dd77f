"""GPU: the sharded PCB and DARE merges (mergerec_b200/merger/sharded.py, `mr_pcb_vectors_dist`) against the single-GPU
`get_pcb_vectors` / `merge_pcb` / `merge_dare`, bit for bit.

* emulated ranks on one GPU: one `DistPcb` per rank, the all-reduces played by hand (sum / max of the workspace views);
  the concatenated slices must equal the single-GPU vectors and merge, over world sizes, model counts, the fast and the
  dense search, forced IEEE divides, quantised inputs, a rank whose updates are all zero, a d mod 32 tail on the last
  rank, empty ranks, and an input whose ranges need the IEEE rerun;
* world 1 (no collective) through `get_pcb_vectors_sharded`, also at BLaIR-base size next to an emulated world 8;
* two processes sharing this GPU (gloo for the collectives): `ShardedModelMerger.merge("pcb" | "dare")` equals
  `ModelMerger.merge`;
* >= 2 GPUs over NCCL (tests/nccl_pcb_worker.py; skipped on one GPU)."""
import multiprocessing as mp
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist

from mergerec_b200 import _lib, synth
from mergerec_b200.merger import ModelMerger
from mergerec_b200.merger.algorithms._common import merge_axpy, weights_tensor
from mergerec_b200.merger.algorithms.pcb import get_pcb_vectors, merge_pcb, pcb_clamp_ranks
from mergerec_b200.merger.sharded import (DistPcb, ShardedModelMerger, flat_shard_bounds, gather_flat, get_pcb_vectors_sharded,
                                          merge_dare_sharded, merge_pcb_sharded)
from test_sharded_merger_host import _free_port

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _bits(t):
    return t.contiguous().view(torch.int32)


def _emulated_clamps(fb, fm, world):
    """The magnitude clamps through emulated `DistSelect` ranks (None where a sampled bracket cannot resolve the input:
    the product path then takes the exact search)."""
    from test_sharded_merger_gpu import _emulated_dist_select
    d = fb.numel()
    i_lo, i_hi = pcb_clamp_ranks(d)
    out = []
    for k in (d - i_lo, d - i_hi):
        if i_lo == 0 or k >= d:
            return None
        sels = _emulated_dist_select(fb, fm, k, world)
        if any(s.status.cpu().tolist() != [1] * len(fm) for s in sels):
            return None
        out.append(torch.stack([(s.cut_global >> 32).to(torch.int32) for s in sels]))
    return [o.view(torch.float32) for o in out]


def _emulated_pcb(fb, fm, density, world, lo, hi, flags=0):
    """`world` DistPcb instances over the slices of one GPU, the collectives played by hand and the host's rerun rule of
    get_pcb_vectors_sharded; returns the ranks and the flags of the last search."""
    d = fb.numel()
    q_index = int(d * (1 - density))
    ranks = []
    for r in range(world):
        a, b = flat_shard_bounds(d, world, r)
        ranks.append(DistPcb(fb[a:b].clone(), [m[a:b].clone() for m in fm], d, a))

    def search(fl):
        for p in ranks:
            p.set_flags(fl)
        for phase, coll in enumerate(ranks[0].collectives):
            for p in ranks:
                p.run(phase, lo, hi, q_index)
            if coll & _lib.MR_PCB_SUM:
                total = torch.stack([p.sum for p in ranks]).sum(0, dtype=torch.int32)
                for p in ranks:
                    p.sum.copy_(total)
            if coll & _lib.MR_PCB_MAX:
                top = torch.stack([p.max for p in ranks]).amax(0)
                for p in ranks:
                    p.max.copy_(top)
        sts = [p.status.cpu().tolist() for p in ranks]
        assert all(s == sts[0] for s in sts), f"ranks disagree on the status: {sts}"
        return sts[0]

    st = search(flags)
    for _ in range(2):
        if st == [1] * len(fm):
            break
        if 0 in st:
            flags |= _lib.MR_PCB_DENSE
        if 2 in st:
            flags |= _lib.MR_PCB_IEEE
        st = search(flags)
    assert st == [1] * len(fm), st
    return ranks, flags


def _check_emulated(base, models, density, world, force_dense=False, force_ieee=False, weights=None):
    fb, fm = dev(base), [dev(m) for m in models]
    K, d = len(fm), fb.numel()
    want, _, _, lo, hi = get_pcb_vectors(fb, fm, density=density, return_diagnostics=True, force_dense=force_dense,
                                         force_ieee=force_ieee)
    ecl = _emulated_clamps(fb, fm, world)
    if ecl is not None:
        for r in range(world):
            assert torch.equal(_bits(ecl[0][r]), _bits(lo)) and torch.equal(_bits(ecl[1][r]), _bits(hi)), f"rank {r}: clamps"
    flags = (_lib.MR_PCB_DENSE if force_dense else 0) | (_lib.MR_PCB_IEEE if force_ieee else 0)
    ranks, used = _emulated_pcb(fb, fm, density, world, lo, hi, flags)
    weights = weights or [0.3 + 0.05 * k for k in range(K)]
    merged = merge_pcb(fb, fm, weights, density=density)
    for r, p in enumerate(ranks):
        a, b = flat_shard_bounds(d, world, r)
        assert torch.equal(_bits(p.out[:, :b - a]), _bits(want[:, a:b])), f"rank {r}: PCB vectors"
        if b > a:
            part = merge_axpy(p.base, list(p.out.unbind(0)), weights_tensor(weights, "cuda"), _lib.MR_ORDER_BASE_FIRST, False)
            assert torch.equal(_bits(part), _bits(merged[a:b])), f"rank {r}: merge_pcb slice"
    return used


FAST, DENSE_D = 1_000_003, 50_021


@pytest.mark.parametrize("world,K", [(2, 1), (3, 3), (4, 8), (8, 16), (2, 16), (8, 3)])
@pytest.mark.parametrize("d", [FAST, DENSE_D])
def test_emulated_ranks_equal_single_gpu(world, K, d):
    base, models = synth.make_flat(d, K, seed=60 + K + world)
    _check_emulated(base, models, 0.2, world)


@pytest.mark.parametrize("world,K,d,dense,ieee", [(4, 8, FAST, True, False), (3, 5, FAST, False, True),
                                                   (2, 3, DENSE_D, True, True), (8, 8, FAST, True, True)])
def test_emulated_forced_dense_and_ieee(world, K, d, dense, ieee):
    base, models = synth.make_flat(d, K, seed=7)
    used = _check_emulated(base, models, 0.2, world, force_dense=dense, force_ieee=ieee)
    assert bool(used & _lib.MR_PCB_DENSE) == dense and bool(used & _lib.MR_PCB_IEEE) == ieee


@pytest.mark.parametrize("world,K,d,quant,density", [(4, 8, FAST, 1e-4, 0.2), (3, 5, DENSE_D, 2.5e-4, 0.2),
                                                      (2, 3, FAST, 5e-4, 0.5)])
def test_emulated_quantised_inputs(world, K, d, quant, density):
    """Many equal task values and magnitudes at the clamps: the order statistics are exact, ties included."""
    base, models = synth.make_flat(d, K, seed=17, quantize=quant)
    _check_emulated(base, models, density, world)


@pytest.mark.parametrize("d", [FAST, DENSE_D])
def test_emulated_rank_with_all_zero_updates(d):
    world, K = 3, 4
    base, models = synth.make_flat(d, K, seed=23)
    a, b = flat_shard_bounds(d, world, 1)
    for m in models:
        m[a:b] = base[a:b]
    _check_emulated(base, models, 0.2, world)


@pytest.mark.parametrize("world,K,d", [(3, 6, 1_000_034), (4, 5, 50_018), (2, 16, 131_106)])
def test_emulated_tail_on_the_last_rank(world, K, d):
    """d mod 32 = 2 with K >= 5 (Recformer-like): the interleaved torch.sum(dim=0) order of the tail on the last rank."""
    assert d % 32 == 2
    base, models = synth.make_flat(d, K, seed=31)
    _check_emulated(base, models, 0.2, world)


@pytest.mark.parametrize("world,K,d", [(8, 3, 200), (8, 5, 64), (5, 2, 100), (3, 4, 1), (2, 2, 2)])
def test_emulated_tiny_vectors_and_empty_ranks(world, K, d):
    """d = 200 / 64 over 8 ranks leaves ranks without columns; d < 100 has i_lo == 0."""
    base, models = synth.make_flat(d, K, seed=37)
    _check_emulated(base, models, 0.2, world)


def test_emulated_degenerate_ranges_rerun_with_ieee_divides():
    """The input of test_degenerate_ranges_fall_back_to_ieee_divides: status 2 on every rank, every rank reruns with IEEE
    divides, and the result equals the single-GPU one."""
    K, d = 3, 200_003
    rng = np.random.default_rng(5)
    base = rng.standard_normal(d).astype(np.float32) * np.float32(1e-20)
    models = [(base + rng.standard_normal(d).astype(np.float32) * np.float32(1e-25)).astype(np.float32) for _ in range(K)]
    used = _check_emulated(base, models, 0.2, 3)
    assert used & _lib.MR_PCB_IEEE


@pytest.mark.parametrize("d,K,quant,density", [(FAST, 8, 0.0, 0.2), (DENSE_D, 3, 2.5e-4, 0.1), (64, 3, 0.0, 0.2),
                                                (200, 5, 0.0, 0.2), (2, 2, 0.0, 0.2)])
def test_world1_matches_single_gpu(d, K, quant, density):
    base, models = synth.make_flat(d, K, seed=3, quantize=quant)
    fb, fm = dev(base), [dev(m) for m in models]
    want = get_pcb_vectors(fb, fm, density=density)
    got = get_pcb_vectors_sharded(fb, fm, density, d)
    assert torch.equal(_bits(got[:, :d]), _bits(want[:, :d]))
    w = [0.2 + 0.1 * k for k in range(K)]
    assert torch.equal(_bits(merge_pcb_sharded(fb, fm, w, density, d)), _bits(merge_pcb(fb, fm, w, density=density)))


def test_world1_degenerate_ranges():
    K, d = 3, 200_003
    rng = np.random.default_rng(5)
    base = rng.standard_normal(d).astype(np.float32) * np.float32(1e-20)
    models = [(base + rng.standard_normal(d).astype(np.float32) * np.float32(1e-25)).astype(np.float32) for _ in range(K)]
    fb, fm = dev(base), [dev(m) for m in models]
    assert torch.equal(_bits(get_pcb_vectors_sharded(fb, fm, 0.2, d)[:, :d]), _bits(get_pcb_vectors(fb, fm, density=0.2)[:, :d]))


def test_blair_base_world1_and_emulated_world8():
    """BLaIR-base size (d = 124,645,632), K = 8: world 1 and 8 emulated ranks give the single-GPU vectors."""
    d, K = synth.total_numel(synth.roberta_shapes()), 8
    g = torch.Generator(device="cuda").manual_seed(3)
    base = torch.randn(d, generator=g, device="cuda") * 0.02
    models = [base + 1e-3 * torch.randn(d, generator=g, device="cuda") for _ in range(K)]
    want, _, _, lo, hi = get_pcb_vectors(base, models, density=0.2, return_diagnostics=True)
    got = get_pcb_vectors_sharded(base, models, 0.2, d)
    assert torch.equal(_bits(got[:, :d]), _bits(want[:, :d]))
    del got
    ranks, used = _emulated_pcb(base, models, 0.2, 8, lo, hi)
    assert used == 0                                  # the fast search on every rank, no rerun
    for r, p in enumerate(ranks):
        a, b = flat_shard_bounds(d, 8, r)
        assert torch.equal(_bits(p.out[:, :b - a]), _bits(want[:, a:b])), f"rank {r}"


# ------------------------------------------------------------------------------------- two processes on one GPU (gloo)
def _state_dicts(recformer):
    shapes = synth.tiny_shapes(recformer=recformer)
    base, models = synth.make_state_dicts(shapes, 5, seed=22 if recformer else 8, sigma=1e-2)
    to_t = lambda sd: {k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}  # noqa: E731
    return to_t(base), [to_t(m) for m in models]


def _same(a, b):
    return list(a.keys()) == list(b.keys()) and all(torch.equal(a[k], b[k]) for k in a)


def _merger_checks(group, world, rank):
    bad = []
    for recformer in (False, True):
        base, models = _state_dicts(recformer)
        ref = ModelMerger(models, base)
        sh = ShardedModelMerger(models, base, group=group)
        tag = "recformer" if recformer else "roberta"
        for w, dens in ((0.3, 0.2), ([0.1, 0.5, 0.2, 0.3, 0.4], 0.1)):
            if not _same(ref.merge("pcb", w, density=dens), sh.merge("pcb", w, density=dens)):
                bad.append(f"{tag}:pcb:{dens}")
        d = ref.models[0].numel()
        for p in (0.1, 0.0, 1.0):
            gm = torch.Generator(device="cpu").manual_seed(5)
            masks = torch.rand((5, d), generator=gm) >= p           # on the host: each rank copies its columns
            if not _same(ref.merge("dare", 0.4, density=p, masks=masks), sh.merge("dare", 0.4, density=p, masks=masks)):
                bad.append(f"{tag}:dare-masks:{p}")
            masks_dev = masks.cuda()                                  # on the device: read in place
            if not _same(ref.merge("dare", 0.4, density=p, masks=masks_dev), sh.merge("dare", 0.4, density=p, masks=masks_dev)):
                bad.append(f"{tag}:dare-masks-dev:{p}")
        a = ref.merge("dare", 0.4, density=0.3, generator=torch.Generator(device="cuda").manual_seed(99))
        b = sh.merge("dare", 0.4, density=0.3, generator=torch.Generator(device="cuda").manual_seed(99))
        if not _same(a, b):
            bad.append(f"{tag}:dare-seeded")
    # flat vectors through the functions: d < 100 (the row-minimum clamp), a ragged split, the fast search
    for d, K in ((64, 3), (200, 4), (300_007, 5)):
        base, models = synth.make_flat(d, K, seed=d)
        fb, fm = dev(base), [dev(m) for m in models]
        lo, hi = flat_shard_bounds(d, world, rank)
        want = get_pcb_vectors(fb, fm, density=0.2)
        got = get_pcb_vectors_sharded(fb[lo:hi].clone(), [m[lo:hi].clone() for m in fm], 0.2, d, group)
        if not torch.equal(_bits(got[:, :hi - lo]), _bits(want[:, lo:hi])):
            bad.append(f"flat:{d}:vectors")
        w = [0.5] * K
        m = merge_pcb_sharded(fb[lo:hi].clone(), [m[lo:hi].clone() for m in fm], w, 0.2, d, group)
        if not torch.equal(_bits(gather_flat(m, d, group)), _bits(merge_pcb(fb, fm, w, density=0.2))):
            bad.append(f"flat:{d}:merge")
        masks = torch.rand((K, d), device="cuda") >= 0.2
        from mergerec_b200.merger.algorithms.dare import merge_dare
        m = merge_dare_sharded(fb[lo:hi].clone(), [m[lo:hi].clone() for m in fm], w, 0.2, d, masks=masks, group=group)
        full = merge_dare(fb, fm, w, 0.2, masks=masks)
        if not torch.equal(_bits(m), _bits(full[lo:hi])):
            bad.append(f"flat:{d}:dare")
    return bad


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.cuda.set_device(0)
        torch.manual_seed(1234)           # the same random masks on both ranks
        q.put((rank, _merger_checks(dist.group.WORLD, world, rank)))
    except Exception as e:  # noqa: BLE001
        import traceback
        q.put((rank, repr(e) + traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def test_two_ranks_on_one_gpu_model_merger_pcb_and_dare():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert sorted(results) == [(0, []), (1, [])]


# ------------------------------------------------------------------------------------------------ NCCL, >= 2 GPUs
def test_sharded_pcb_and_dare_over_nccl():
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import nccl_pcb_worker
        assert nccl_pcb_worker.main() == 0
        return
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (or a torchrun launch with WORLD_SIZE > 1)")
    for g in sorted({2, min(n, 8)}):
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={g}", "--master-addr",
               "127.0.0.1", "--master-port", str(_free_port()), os.path.join(HERE, "nccl_pcb_worker.py")]
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, (g, out.stdout[-2000:], out.stderr[-4000:])
        assert f"nccl pcb worker: ok (world {g})" in out.stdout
