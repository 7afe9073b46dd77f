"""GPU: the PCB quantile search (csrc/pcb.cu) against exact order statistics, on inputs built to break it.

The fast search finds the int(d (1 - density))-th smallest balancing weight of every model from a 1/32 sample at hashed
positions, a key window of +-R sample ranks, one pass that counts the keys below the window and collects the keys inside
it in per-warp lists, and three refinement levels over those lists.  A window that misses the rank or a list that
overflows must be reported (status 0) and redone by the three dense radix passes; a range outside [2^-60, 2^60] must be
reported (status 2) and redone with IEEE divides.  Every case here is checked against references that do not use the
kernel's search:

1. the 1 % / 99 % magnitude clamps, bit for bit, against a host sort of |tau_k|;
2. the quantile and the row maximum against a host sort of the kernel's own balancing weights (by value: -0 == +0,
   NaN == NaN);
3. the balancing weights against the numpy oracle (4e-7 relative);
4. the vectors: equal as values (+-0 and NaN payloads aside) to pcb.py's formula evaluated in fp32 on the kernel's own
   balancing weights; against the
   oracle at 2e-6 of the row scale plus the first-order effect of the weights' libm differences on the clamped scales,
   excluding only columns where a balancing weight differs from the threshold by a nonzero amount within 1e-3 relative
   (a few denormal ulp when the threshold is 0): weights equal to the threshold are clamped to the same value on both
   sides and stay in;
5. the same bits from the forced dense search and, where nothing needed a rerun, from forced IEEE divides;
6. the per-model status of one `mr_pcb_vectors` call with flags = 0: a model that reports 1 carries the exact key.

Input families: Gaussian updates (control), bf16-rounded checkpoints, columns frozen in every model (a tie of +0 keys
around the quantile), models paired as tau / -tau (a mix of +0 and -0 keys), large updates planted at exactly the
sampled quads of one model (the window misses) and next to them (it does not), ranges at the edges of [2^-60, 2^60],
and models equal to the base (range 0: the reference's normalisation is 0 / 0, every vector NaN)."""
import time

import numpy as np
import pytest
import torch
from hypothesis import example, given, settings, strategies as st

from mergerec_b200 import _lib, synth
from mergerec_b200.merger import ModelMerger
from mergerec_b200.merger.algorithms._common import as_rows
from mergerec_b200.merger.algorithms.pcb import get_pcb_vectors, merge_pcb, pcb_clamp_ranks
from mergerec_b200.merger.layout import FlatLayout, alloc_rows
from mergerec_b200.merger.sharded import DistPcb, flat_shard_bounds, get_pcb_vectors_sharded
from oracle import oracle as orc
from test_property_gpu import SETTINGS, shifted
from test_sharded_pcb_gpu import _check_emulated

pytestmark = pytest.mark.gpu

STRIDE = 32                  # pcb.cu kPcbStride: the fast path samples one quad out of every 4 * STRIDE columns
FIRST_FAST = 4096 * STRIDE   # d = 131,072: the first size with pcb_sample_count(d) >= 4096
PLANT = np.float32(0.05)     # a planted update: 50 sigma of synth.make_flat's updates
TOL = 2e-6


def host(t):
    return t.detach().cpu().numpy()


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same_value(a, b):
    """Equal as values (-0 == +0), NaN matching NaN."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return bool(((a == b) | (np.isnan(a) & np.isnan(b))).all())


# ---------------------------------------------------------------------------------------------------- input families
def sample_columns(d):
    """numpy mirror of pcb_sample_column over the whole sample: quad c sits at 4 * (hash(c) % 32) in block c of 128."""
    n_s = 4 * (d // (4 * STRIDE))
    i = np.arange(n_s, dtype=np.int64)
    c = i >> 2
    h = ((c.astype(np.uint64) * np.uint64(2654435761)) & np.uint64(0xFFFFFFFF)) >> np.uint64(16)
    return c * (4 * STRIDE) + 4 * (h % np.uint64(STRIDE)).astype(np.int64) + (i & 3)


def planted_columns(d, control=False):
    """Every fourth sampled quad (one in 512 columns): enough to move the sample's order statistics far past the window's
    +-6 sigma, too few to move the quantile of the whole vector.  control: the same quads moved 4 columns inside their
    block, off the sample."""
    cols = sample_columns(d).reshape(-1, 4)[::4].reshape(-1)
    if control:
        cols = cols + np.where((cols % (4 * STRIDE)) // 4 == STRIDE - 1, -4, 4)
    return cols


def frozen_mask(rng, d, f):
    """f * d columns: about 80 % of them as tensor-sized runs of 6144 (8 rows of 768), the rest scattered."""
    n, run = int(round(f * d)), 768 * 8
    mask = np.zeros(d, bool)
    for s in rng.choice(d // run, size=int(0.8 * n) // run, replace=False):
        mask[s * run:(s + 1) * run] = True
    mask[rng.choice(np.flatnonzero(~mask), size=n - int(mask.sum()), replace=False)] = True
    return mask


def frozen_edge_mask(rng, base, models, q_index, edge):
    """Columns to freeze so that model 0's q_index-th smallest balancing weight is the LAST element of the tie of +0
    weights (edge = 'hi') or its FIRST (edge = 'lo').  The sign of tanh(tau_0 * sum tau) is that of the fp32 product, so
    the count of negative and of zero weights in the unfrozen columns is known on the host.  Columns are frozen in a fixed
    order -- 6144-column runs first, then single columns -- and the order is cut where the count is exact."""
    d = base.size
    tau = (np.stack(models) - base[None, :]).astype(np.float32)
    prod = (tau[0] * orc._sum_dim0(tau)).astype(np.float32)
    run = 768 * 8
    runs = rng.permutation(d // run)
    in_runs = (runs[:, None] * run + np.arange(run)[None, :]).reshape(-1)
    rest = np.setdiff1d(np.arange(d), in_runs)
    order = np.concatenate([in_runs, rng.permutation(rest)])
    neg, zero = (prod < 0)[order], (prod == 0)[order]
    n = np.arange(d + 1)
    below = int((prod < 0).sum()) - np.concatenate([[0], np.cumsum(neg)])     # negative weights left after freezing n
    tie = n + int((prod == 0).sum()) - np.concatenate([[0], np.cumsum(zero)])  # +-0 weights after freezing n
    hit = np.flatnonzero(below + tie == q_index + 1) if edge == "hi" else np.flatnonzero((below == q_index) & (tie > 0))
    assert hit.size, (edge, q_index)
    mask = np.zeros(d, bool)
    mask[order[:hit[0]]] = True
    return mask


def tie_position(task, q_index):
    """Where rank q_index falls relative to the tie of zero weights of each row: 'above', 'below', 'first', 'last',
    'inside' (strictly between its ends)."""
    out = []
    for t in task:
        lt, eq = int((t < 0).sum()), int((t == 0).sum())
        if q_index < lt:
            out.append("below")
        elif q_index >= lt + eq:
            out.append("above")
        else:
            out.append("first" if q_index == lt else "last" if q_index == lt + eq - 1 else "inside")
    return out


def _bf16(x):
    return torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(torch.bfloat16).to(torch.float32).numpy()


def _range_edge(d, K, seed, kind):
    """base = 0, so tau_k = m_k exactly; each model is scaled so that its clamp range hi - lo lies just inside ('lo_in')
    or just outside ('lo_out') 2^-60, or its upper clamp hi (and with it the range) just inside / outside 2^60.  The low
    kinds plant |tau| = 1 in 0.5 % of the columns of every model (above the 99 % clamp), which keeps the span of the
    balancing weights far inside the range."""
    rng = np.random.default_rng(seed)
    base = np.zeros(d, np.float32)
    top = rng.choice(d, size=d // 200, replace=False) if kind.startswith("lo") else None
    i_lo, i_hi = pcb_clamp_ranks(d)
    models = []
    for _ in range(K):
        g = rng.standard_normal(d).astype(np.float64)
        if top is not None:
            g[top] = 1e30
        mag = np.sort(np.abs(g))
        glo, ghi = mag[i_lo], mag[i_hi]
        edge, nudge = {"lo_in": (2.0 ** -60, 1 + 2 ** -8), "lo_out": (2.0 ** -60, 1 - 2 ** -8),
                       "hi_in": (2.0 ** 60, 1 - 2 ** -8), "hi_out": (2.0 ** 60, 1 + 2 ** -8)}[kind]
        s = edge * nudge / ((ghi - glo) if kind.startswith("lo") else ghi)
        m = (g * s).astype(np.float32)
        if top is not None:
            m[top] = 1.0
        models.append(m)
    # the predicate of pcb_safe_range, on the clamps the kernels will read
    for m in models:
        mag = np.sort(np.abs(m))
        lo, hi = mag[i_lo], mag[i_hi]
        rng_ = np.float32(hi - lo)
        inside = (2.0 ** -60 <= rng_ <= 2.0 ** 60) and (2.0 ** -60 <= hi <= 2.0 ** 60)
        assert inside == kind.endswith("_in"), (kind, lo, hi)
    return base, models


def make_case(family, d, K, seed, density=0.2):
    """(base, models) of one family.  The planted families plant into model 0; 'frozen:edge_hi' / 'frozen:edge_lo' put
    model 0's quantile at the upper / lower end of the tie of frozen columns for this density."""
    name, _, arg = family.partition(":")
    if name == "range_edge":
        return _range_edge(d, K, seed, arg)
    base, models = synth.make_flat(d, K, seed=seed)
    rng = np.random.default_rng(seed + 1000)
    if name == "bf16grid":
        base, models = _bf16(base), [_bf16(m) for m in models]
    elif name == "frozen":
        if arg.startswith("edge"):
            mask = frozen_edge_mask(rng, base, models, int(d * (1 - density_for(d, density))), arg[5:])
        else:
            mask = frozen_mask(rng, d, float(arg))
        for m in models:
            m[mask] = base[mask]
    elif name == "cancel":
        cols = rng.random(d) < 0.5
        for k in range(0, K - 1, 2):
            t = (models[k] - base).astype(np.float32)
            m1 = (base - t).astype(np.float32)
            sel = cols & ((m1 - base).astype(np.float32) == -t)     # where tau_{k+1} = -tau_k exactly
            models[k + 1][sel] = m1[sel]
    elif name in ("planted_high", "planted_control"):
        cols = planted_columns(d, control=name == "planted_control")
        models[0][cols] = (base[cols] + PLANT).astype(np.float32)
    elif name == "planted_low":
        cols = sample_columns(d)                # the whole sample of model 0 at +0, far below the 80 % quantile
        models[0][cols] = base[cols]
    elif name == "base_model":
        for k in range(K if arg == "all" else 1):
            models[k] = base.copy()
    else:
        assert name == "gauss", family
    return base, models


def density_for(d, density):
    """'last': the density with int(d (1 - density)) = d - 1 (the window's open upper end)."""
    if density == "last":
        density = 0.5 / d
        assert int(d * (1 - density)) == d - 1
    return density


# ---------------------------------------------------------------------------------------------------- the checks
def search_status(tb, tm, lo, hi, q_index):
    """One `mr_pcb_vectors` call with flags = 0 (built like get_pcb_vectors' `run`): per-model status, task, thresholds."""
    lib = _lib.load()
    rows = as_rows(tm)
    K, d = len(rows), tb.numel()
    out, task = alloc_rows(K, d, tb.device), alloc_rows(K, d, tb.device)
    thr = torch.empty((K, 2), dtype=torch.float32, device=tb.device)
    ws_bytes = int(lib.mr_pcb_workspace_bytes(d, K))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=tb.device)
    status = torch.full((K,), -1, dtype=torch.int32, device=tb.device)
    rc = lib.mr_pcb_vectors(_lib.dptr(tb, torch.float32), _lib.ptr_array(rows), K, d, _lib.dptr(lo), _lib.dptr(hi), q_index,
                            0, _lib.dptr(status), _lib.dptr(out), max(out.stride(0), d), _lib.dptr(task), _lib.dptr(thr),
                            _lib.dptr(ws), ws_bytes, _lib.stream_handle())
    _lib.check(rc, "mr_pcb_vectors")
    return host(status), host(task), host(thr)


def near_threshold(task, q):
    """Columns where some model's weight differs from its threshold by a NONZERO amount within 1e-3 relative (4 denormal
    ulp when the threshold is 0): there an ulp of libm difference can move the weight across the clamp."""
    diff = np.abs(task.astype(np.float64) - q.astype(np.float64)[:, None])
    tol = np.where(q == 0, 4 * 2.0 ** -149, 1e-3 * np.abs(q.astype(np.float64)))[:, None]
    return ((diff > 0) & (diff <= tol)).any(axis=0)


def check_case(family, d, K, density, shift, seed):
    density = density_for(d, density)
    base, models = make_case(family, d, K, seed, density)
    q_index = int(d * (1 - density))
    tb, tm = shifted(base, shift, d), [shifted(m, shift, d) for m in models]
    out, task, thr, lo, hi = get_pcb_vectors(tb, tm, density=density, return_diagnostics=True)
    out_h, task_h, thr_h, lo_h, hi_h = host(out), host(task), host(thr), host(lo), host(hi)
    tag = f"{family} d={d} K={K} density={density} shift={shift}"

    # 1. clamps: exact order statistics of |tau_k|
    mag = np.sort(np.abs(np.stack(models) - base[None, :]), axis=1)
    i_lo, i_hi = pcb_clamp_ranks(d)
    assert np.array_equal(_bits(lo_h), _bits(mag[:, i_lo])) and np.array_equal(_bits(hi_h), _bits(mag[:, i_hi])), tag
    del mag
    # 2. quantile and maximum of the kernel's own balancing weights
    srt = np.sort(task_h, axis=1)
    assert same_value(thr_h[:, 0], srt[:, q_index]), (tag, thr_h[:, 0], srt[:, q_index])
    assert same_value(thr_h[:, 1], srt[:, -1]), (tag, thr_h[:, 1], srt[:, -1])
    del srt
    # 3. balancing weights against the oracle
    o_vec, o_task, o_q, _, o_lo, o_hi = orc.pcb_vectors(base, models, density, return_task=True)
    assert np.array_equal(_bits(lo_h), _bits(o_lo)) and np.array_equal(_bits(hi_h), _bits(o_hi)), tag
    assert np.array_equal(np.isnan(task_h), np.isnan(o_task)), tag
    fin = ~np.isnan(o_task)
    assert (np.abs(task_h[fin].astype(np.float64) - o_task[fin]) <= 4e-7 * np.abs(o_task[fin]) + 1e-44).all(), tag
    # 4a. vectors, exactly: pcb.py:53-56 evaluated in fp32 on the kernel's own balancing weights and thresholds (every
    # column, ties and near-threshold weights included)
    tau = (np.stack(models) - base[None, :]).astype(np.float32)
    A = np.minimum(np.maximum(np.abs(tau), lo_h[:, None]), hi_h[:, None])
    q, mx = thr_h[:, :1], thr_h[:, 1:]
    with np.errstate(invalid="ignore", divide="ignore"):
        scale = ((np.minimum(np.maximum(task_h, q), mx) - q) / (mx - q)).astype(np.float32)
        want = ((np.sign(tau) * A).astype(np.float32) * scale).astype(np.float32)
        want = (want / np.maximum(orc._sum_dim0(scale), np.float32(1e-12))[None, :]).astype(np.float32)
        want = (want / np.float32(K)).astype(np.float32)
    assert same_value(out_h, want), (tag, int((~((out_h == want) | (np.isnan(out_h) & np.isnan(want)))).sum()), "columns differ")
    del tau, A, scale, want
    # 4b. vectors against the oracle: NaN exactly where it has NaN; elsewhere within 2e-6 of the row scale plus the
    # first-order effect of the balancing weights' libm differences (1e-6 relative, twice the bound of check 3) on the
    # scales (t - q) / (max - q): the normalised vector moves by at most twice the largest relative change of a scale in
    # its column.  Columns with a weight a NONZERO amount within 1e-3 relative of its threshold are excluded (there the
    # clamp is discontinuous); weights equal to the threshold are not.
    assert np.array_equal(np.isnan(out_h), np.isnan(o_vec)), (tag, int(np.isnan(out_h).sum()), int(np.isnan(o_vec).sum()))
    near = near_threshold(task_h, thr_h[:, 0]) | near_threshold(o_task, o_q)
    compared = d - int(near.sum())
    assert near.sum() <= max(0.01 * d, 2 * K), (tag, f"{compared} of {d} columns compared")
    gap = o_task.astype(np.float64) - o_q.astype(np.float64)[:, None]
    with np.errstate(invalid="ignore", divide="ignore"):
        cond = np.where(gap > 0, 1e-6 * (np.abs(o_task) + np.abs(o_q)[:, None]) / gap, 0.0)
    cond = np.nan_to_num(cond, nan=0.0).max(axis=0)
    for k in range(K):
        ok = ~near & ~np.isnan(o_vec[k])
        if ok.any():
            row = max(float(np.abs(o_vec[k][ok]).max()), 1e-37)
            err = np.abs(out_h[k][ok].astype(np.float64) - o_vec[k][ok])
            bound = TOL * row + 2 * cond[ok] * np.abs(o_vec[k][ok])
            assert (err <= bound).all(), (tag, k, float((err / row).max()), f"{compared} of {d} columns compared")
    # 5. the forced dense search and forced IEEE divides give the same bits
    dense, _, thr_d, *_ = get_pcb_vectors(tb, tm, density=density, return_diagnostics=True, force_dense=True)
    assert np.array_equal(_bits(host(dense)), _bits(out_h)) and np.array_equal(_bits(host(thr_d)), _bits(thr_h)), tag
    # 6. status of the search with flags = 0
    status, task_s, thr_s = search_status(tb, tm, lo, hi, q_index)
    assert set(status.tolist()) <= {0, 1, 2}, (tag, status)
    srt = np.sort(task_s, axis=1)
    for k in np.flatnonzero(status == 1):
        assert same_value(thr_s[k, 0], srt[k, q_index]) and same_value(thr_s[k, 1], srt[k, -1]), (tag, k, "wrong key, status 1")
    if (status == 1).all():
        ieee = get_pcb_vectors(tb, tm, density=density, force_ieee=True)
        assert np.array_equal(_bits(host(ieee)), _bits(out_h)), tag
    return dict(status=status, out=out_h, o_vec=o_vec, task=task_h, thr=thr_h, q_index=q_index)


def expected_status(family, d, density, status):
    """The status words a family must produce on the fast path."""
    name, _, arg = family.partition(":")
    if d < FIRST_FAST:
        assert (status != 0).all(), status                  # the dense search never misses
        return
    if name in ("gauss", "planted_control", "bf16grid", "cancel") or (name == "range_edge" and arg.endswith("_in")):
        # q_index = d - 1: the quantile is the row maximum, the span max - q is 0 (the reference's 0 / 0) -> IEEE divides
        want = 2 if int(d * (1 - density_for(d, density))) == d - 1 else 1
        assert (status == want).all(), (family, status)
    elif name in ("planted_high", "planted_low"):
        assert status[0] == 0, (family, status)            # the planted model's window misses: reported, not returned
    elif name == "range_edge":
        assert (status == 2).all(), (family, status)


LAST = "last"
CASES = [
    # family,            d,          K,  density, shift
    ("gauss",            131_072,    1,  0.2,     0),
    ("gauss",            131_071,    2,  0.2,     0),       # the last dense size
    ("gauss",            1_000_003,  16, 0.2,     1),
    ("gauss",            600_011,    7,  1.0,     0),       # q_index = 0: the window's open lower end
    ("gauss",            131_199,    7,  LAST,    2),       # unsampled partial block; q_index = d - 1
    ("gauss",            600_011,    2,  1e-3,    0),
    ("gauss",            600_011,    5,  0.999,   3),
    ("bf16grid",         131_072,    16, 0.2,     0),
    ("bf16grid",         1_000_003,  7,  0.5,     3),
    ("bf16grid",         600_011,    1,  LAST,    0),
    ("frozen:0.5",       600_011,    8,  0.2,     0),
    ("frozen:0.79",      600_011,    8,  0.2,     0),
    ("frozen:0.80",      1_000_003,  5,  0.2,     1),
    ("frozen:0.81",      131_072,    16, 0.2,     0),
    ("frozen:0.95",      600_011,    3,  0.2,     2),
    ("frozen:0.80",      131_199,    1,  1.0,     0),
    ("frozen:edge_hi",   600_011,    8,  0.2,     0),
    ("frozen:edge_hi",   131_072,    16, 0.2,     3),
    ("frozen:edge_lo",   1_000_003,  8,  0.7,     1),
    ("cancel",           600_011,    4,  0.2,     0),
    ("cancel",           1_000_003,  16, 1.0,     2),
    ("cancel",           131_072,    2,  LAST,    0),
    ("planted_high",     600_011,    4,  0.2,     0),
    ("planted_high",     131_072,    1,  0.2,     1),
    ("planted_low",      600_011,    3,  0.2,     0),
    ("planted_low",      1_000_003,  16, 0.5,     0),
    ("planted_control",  600_011,    4,  0.2,     0),
    ("planted_control",  131_072,    1,  0.2,     1),
    ("range_edge:lo_in",  200_003,   3,  0.2,     0),
    ("range_edge:lo_out", 200_003,   3,  0.2,     0),
    ("range_edge:hi_in",  200_003,   3,  0.2,     1),
    ("range_edge:hi_out", 200_003,   3,  0.2,     1),
    ("base_model:one",   600_011,    3,  0.2,     0),
    ("base_model:all",   131_072,    1,  0.2,     0),
]


# where the quantile rank falls relative to the tie of +0 weights that frozen columns make: every model, or model 0 for
# the edge constructions (the other models' ties end elsewhere)
TIE_POSITION = {"frozen:0.5": "above", "frozen:0.79": "inside", "frozen:0.80": "inside", "frozen:0.81": "inside",
                "frozen:0.95": "inside", "frozen:edge_hi": "last", "frozen:edge_lo": "first"}


@pytest.mark.parametrize("family,d,K,density,shift", CASES, ids=[f"{c[0]}-d{c[1]}-K{c[2]}-{c[3]}-s{c[4]}" for c in CASES])
def test_search_against_exact_order_statistics(family, d, K, density, shift):
    res = check_case(family, d, K, density, shift, seed=d % 1000 + K)
    expected_status(family, d, density, res["status"])
    if family.startswith("frozen"):
        pos = tie_position(res["task"], res["q_index"])
        want = TIE_POSITION[family] if K > 1 else "first"          # K = 1: no negative weights, the tie starts at rank 0
        assert (pos[0] == want) if "edge" in family else (pos == [want] * K), (family, pos)
    if family.startswith("base_model"):
        # the rows equal to the base have NaN balancing weights (IEEE 0 / 0): their quantile and maximum are NaN too
        assert np.isnan(res["thr"][0]).all(), res["thr"]
        assert np.isnan(res["o_vec"]).all() and np.isnan(res["out"]).all()


@pytest.mark.parametrize("which", ["one", "all"])
def test_models_equal_to_the_base_give_nan_everywhere(which):
    """Range 0: pcb.py's normalisation is 0 / 0, so every column of every vector is NaN.  The fast divisions report
    status 2 and the call reruns with IEEE divides; no entry point may raise, and each must return NaN exactly where the
    oracle has NaN."""
    d, K, density = 600_011, 3, 0.2
    base, models = make_case(f"base_model:{which}", d, K, seed=5)
    o_vec = orc.pcb_vectors(base, models, density)
    assert np.isnan(o_vec).all()
    tb, tm = torch.from_numpy(base).cuda(), [torch.from_numpy(m).cuda() for m in models]
    assert np.isnan(host(get_pcb_vectors(tb, tm, density=density))).all()
    assert np.isnan(host(get_pcb_vectors_sharded(tb, tm, density, d))).all()
    w = [0.3] * K
    o_merged = orc.merge_pcb(base, models, w, density)
    merged = host(merge_pcb(tb, tm, w, density=density))
    assert np.array_equal(np.isnan(merged), np.isnan(o_merged)) and np.isnan(merged).all()
    split = 250_000                                                   # two tensors in the state dict
    sd = lambda v: {"a.weight": torch.from_numpy(v[:split].reshape(500, 500)), "b.weight": torch.from_numpy(v[split:])}  # noqa: E731
    out = ModelMerger([sd(m) for m in models], sd(base)).merge("pcb", w, density=density)
    flat = torch.cat([v.reshape(-1).float().cpu() for v in out.values()]).numpy()
    assert flat.shape == (d,) and np.isnan(flat).all()


# ---------------------------------------------------------------------------------------------------- sharded search
@pytest.mark.parametrize("world", [3, 8])
@pytest.mark.parametrize("family", ["bf16grid", "frozen:0.80", "planted_high", "cancel"])
def test_sharded_search_on_the_same_inputs(family, world):
    """The emulated ranks must give the single-GPU vectors bit for bit, which the cases above pin to the oracle."""
    base, models = make_case(family, 600_011, 5, seed=world)
    used = _check_emulated(base, models, 0.2, world)
    if family == "planted_high":
        assert used & _lib.MR_PCB_DENSE, used         # the planted model's miss is reported on every rank


@pytest.mark.parametrize("world", [3, 8])
def test_sharded_sample_blocks_straddling_slice_boundaries(world):
    """Slices start on multiples of 32 columns and sampled blocks span 128, so a block can straddle a boundary; its
    sampled quad must belong to exactly one rank's share of the sample.  Each rank's sample pass must count exactly the
    sampled columns inside its slice (the numpy mirror of pcb_sample_column), and with updates planted at the sampled
    quads next to every boundary the fast sharded search must give the single-GPU vectors without a rerun."""
    d, K = 1_000_003, 4
    base, models = make_case("gauss", d, K, seed=71)
    blocks = []
    for r in range(1, world):
        a = flat_shard_bounds(d, world, r)[0]
        blocks += [a // (4 * STRIDE) - 1, a // (4 * STRIDE), a // (4 * STRIDE) + 1]
    cols = sample_columns(d).reshape(-1, 4)[blocks].reshape(-1)
    models[1][cols] = (base[cols] + PLANT).astype(np.float32)
    fb, fm = torch.from_numpy(base).cuda(), [torch.from_numpy(m).cuda() for m in models]
    _, _, _, lo, hi = get_pcb_vectors(fb, fm, density=0.2, return_diagnostics=True)
    sample = sample_columns(d)
    straddling = 0
    for r in range(world):
        a, b = flat_shard_bounds(d, world, r)
        straddling += int(a % (4 * STRIDE) != 0)
        p = DistPcb(fb[a:b].clone(), [m[a:b].clone() for m in fm], d, a)
        p.run(0, lo, hi, int(d * 0.8))                     # the sample pass: slot-0 histograms of this rank's share
        got = int(p.sum[:K * 2048].to(torch.int64).sum())
        assert got == K * int(((sample >= a) & (sample < b)).sum()), (r, a, b, got)
    assert straddling > 0
    assert _check_emulated(base, models, 0.2, world) == 0


# ---------------------------------------------------------------------------------------------------- randomised
RANDOM_FAMILIES = ["gauss", "bf16grid", "frozen:0.80", "cancel", "planted_high", "planted_control"]
RANDOM_SETTINGS = dict(SETTINGS, max_examples=max(1, SETTINGS["max_examples"] // 8))


@settings(**RANDOM_SETTINGS)
@given(family=st.sampled_from(RANDOM_FAMILIES), d=st.integers(FIRST_FAST, 400_000), K=st.integers(1, 16),
       density=st.sampled_from([1.0, 1e-3, 0.2, 0.5, 0.999, LAST]), shift=st.integers(0, 3), seed=st.integers(0, 2 ** 31 - 1))
@example(family="planted_high", d=FIRST_FAST, K=16, density=0.5, shift=3, seed=1)
def test_random_cases_at_fast_path_sizes(family, d, K, density, shift, seed):
    status = check_case(family, d, K, density, shift, seed)["status"]
    if family in ("gauss", "planted_control") or (family == "planted_high" and density in (0.2, 0.5)):
        expected_status(family, d, density, status)


# ---------------------------------------------------------------------------------------------------- full size
def test_blair_base_bf16_with_frozen_embeddings():
    """BLaIR-base (d = 124,645,632), K = 8, as real checkpoints look: bf16-rounded models, the word embeddings (31 % of
    the columns) and the LayerNorm rows unchanged in every model.  Clamps and quantile against torch.sort row by row;
    the fast entry point and the forced dense search give the same bits."""
    shapes = synth.roberta_shapes()
    lay = FlatLayout.from_shape_dict(shapes)
    d, K, density = lay.d, 8, 0.2
    g = torch.Generator(device="cuda").manual_seed(13)
    base = (torch.randn(d, generator=g, device="cuda") * 0.02).to(torch.bfloat16).float()
    frozen = torch.zeros(d, dtype=torch.bool, device="cuda")
    for name, off, n in zip(lay.names, lay.offsets, lay.sizes):
        if name.endswith("word_embeddings.weight") or ".LayerNorm." in name:
            frozen[off:off + n] = True
    models = [torch.where(frozen, base, (base + 1e-3 * torch.randn(d, generator=g, device="cuda")).to(torch.bfloat16).float())
              for _ in range(K)]
    del frozen
    small = [m[:4096].clone() for m in models]
    get_pcb_vectors(base[:4096].clone(), small, density=density)          # module load and first launches
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out, task, thr, lo, hi = get_pcb_vectors(base, models, density=density, return_diagnostics=True)
    torch.cuda.synchronize()
    print(f"\nget_pcb_vectors, BLaIR-base K=8 bf16 + frozen embeddings: {1e3 * (time.perf_counter() - t0):.1f} ms "
          f"({torch.cuda.get_device_name()})")
    i_lo, i_hi = pcb_clamp_ranks(d)
    q_index = int(d * (1 - density))
    for k in range(K):
        mag = torch.sort((models[k] - base).abs()).values
        assert int(mag[i_lo].view(torch.int32)) == int(lo[k].view(torch.int32)), k
        assert int(mag[i_hi].view(torch.int32)) == int(hi[k].view(torch.int32)), k
        del mag
        srt = torch.sort(task[k, :d]).values
        assert float(srt[q_index]) == float(thr[k, 0]) and float(srt[-1]) == float(thr[k, 1]), k
        del srt
    del task
    dense, _, thr_d, *_ = get_pcb_vectors(base, models, density=density, return_diagnostics=True, force_dense=True)
    assert torch.equal(thr_d.view(torch.int32), thr.view(torch.int32))
    assert torch.equal(dense[:, :d].contiguous().view(torch.int32), out[:, :d].contiguous().view(torch.int32))
