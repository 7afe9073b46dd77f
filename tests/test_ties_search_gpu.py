"""GPU: the TIES sampled-bracket select (csrc/ties.cu) against exact order statistics, on inputs built to break it.

Every TIES-family result depends on one order statistic per model: the int(density d)-th largest composite key
(bits(|w (m - b)|) << 32) | (0xFFFFFFFF - j).  The fast select finds it from a strided sample of about 0.5 M keys (two
looks), one full pass that counts the keys above the bracket and collects the keys inside it in per-thread lists, and
two 1024-way refinements over those lists; `mr_ties_select_build` adds a 4x denser third look and builds the output
with a provisional cut in the same pass.  Whenever the sample lied (the cut lies outside the bracket), a list overflowed
or the refined bracket does not fit the final sort, the model's status word must say so: deferred callers (the CUDA-graph
TIES step, the PCB clamps) trust a result whenever its status is 1.  So the central check here is

    status 1  =>  exactly the reference cut (and, for select + build, exactly the oracle's output),

together with the status each family is built to produce, and the exact results of the public (non-deferred) paths.

References that do not use the kernels' search: the keys rebuilt in numpy and `np.partition` (cross-checked with the C
oracle's select), the oracle's TIES vectors / merge_ties / lambda merge, and a numpy mirror of the sample positions of
`ties_pass_kernel`.  Every family that plants values at sampled positions has a control with the same plants moved off
the sample, which must report 1: together they pin the mirror.

Sizes: d >= 4.2 M makes both the sparse and the dense sample strict subsamples (stride >= 4 quads); d = 3 M only the sparse
one."""
import numpy as np
import pytest
import torch

from mergerec_b200 import _lib, synth
from mergerec_b200.merger.algorithms.ties import (get_ties_vectors, merge_ties, merge_ties_lambda, select_build,
                                                 select_kth_largest)
from mergerec_b200.merger.layout import alloc_rows
from mergerec_b200.merger.sharded import flat_shard_bounds, sharded_select
from oracle import oracle as orc
from test_property_gpu import shifted
from test_sharded_merger_gpu import _emulated_dist_select

pytestmark = pytest.mark.gpu

SAMPLE_QUADS = 131072            # ties.cu kTiesSampleQuads: the sparse sample; mr_ties_select_build's dense one is 4x
DONE, BRACKET_LOW, BRACKET_HIGH, TOO_MANY, CAND_OVERFLOW, INCONSISTENT = 1, -1, -2, -3, -4, -5
STATUSES = {DONE, BRACKET_LOW, BRACKET_HIGH, TOO_MANY, CAND_OVERFLOW, INCONSISTENT}
FAIL = "fail"                    # expected: some status other than 1
PLANT = np.float32(0.05)         # 50 sigma of synth.make_flat's updates: far above every cut


def host(t):
    return t.detach().cpu().numpy()


def cut_u64(t):
    return host(t).view(np.uint64)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ---------------------------------------------------------------------------------------------------- the sample mirror
def sample_stride(d, quads=SAMPLE_QUADS):
    """ties_sample_stride: quads between two picks (even), 1 = every quad."""
    s = (2 * ((d + 3) >> 2) // quads) & ~1
    return 1 if s < 2 else s


def sampled_pairs(d_local, stride):
    """First quads of the picked pairs of ties_pass_kernel over a vector of d_local elements (local quad indices): window
    pos picks q = pos * stride + ((pos * 2654435761 mod 2^32) >> 8) % stride, rounded down to even, and q + 1."""
    nq = (d_local + 3) >> 2
    if stride == 1:
        return np.arange(0, nq, 2, dtype=np.int64)
    pos = np.arange(-(-nq // stride), dtype=np.int64)
    h = ((pos.astype(np.uint64) * np.uint64(2654435761)) & np.uint64(0xFFFFFFFF)) >> np.uint64(8)
    q = (pos * stride + (h % np.uint64(stride)).astype(np.int64)) & ~np.int64(1)
    return q[q < nq]


def pair_columns(pairs, d):
    """The (up to) 8 elements of each pair of quads."""
    cols = (4 * pairs[:, None] + np.arange(8)[None, :]).reshape(-1)
    return cols[cols < d]


def off_sample(pairs, d, avoid):
    """Each pair moved to the nearest pair (+-2, +-4 quads) that is in no sampled set of `avoid`: the control plants."""
    nq = (d + 3) >> 2
    out = np.full(pairs.shape, -1, np.int64)
    for step in (2, -2, 4, -4, 6, -6):
        c = pairs + step
        ok = (out < 0) & (c >= 0) & (c + 1 < nq)
        for a in avoid:
            ok &= ~np.isin(c, a)
        out = np.where(ok, c, out)
    assert (out >= 0).all()
    return np.unique(out)


# ---------------------------------------------------------------------------------------------------- references
def keys_of(base, m, wk=None):
    d = base.size
    with np.errstate(all="ignore"):
        u = (m - base).astype(np.float32)
        if wk is not None:
            u = (u * np.float32(wk)).astype(np.float32)
    mag = (u.view(np.uint32) & np.uint32(0x7FFFFFFF)).astype(np.uint64)
    return (mag << np.uint64(32)) | (np.uint64(0xFFFFFFFF) - np.arange(d, dtype=np.uint64))


def ref_cuts(base, models, k_cnt, w=None):
    """The k_cnt-th largest key of every model (np.partition), cross-checked with the C oracle's select."""
    d = base.size
    out = np.empty(len(models), np.uint64)
    for k, m in enumerate(models):
        if k_cnt <= 0:
            out[k] = np.uint64(0xFFFFFFFFFFFFFFFF)
        elif k_cnt >= d:
            out[k] = 0
        else:
            out[k] = np.partition(keys_of(base, m, None if w is None else w[k]), d - k_cnt)[d - k_cnt]
    return out


def same_survivors(base, models, got, ref, w=None):
    """`sharded_select`'s cut: the canonical key, except that its exact windowed search returns mag << 32 ("every element
    at this magnitude survives") when the reference keeps every element at the cut magnitude.  A partial tie at the cut
    must give the canonical key itself."""
    for k, m in enumerate(models):
        if got[k] != ref[k]:
            mag = ref[k] >> np.uint64(32)
            if got[k] != mag << np.uint64(32):
                return False
            keys = keys_of(base, m, None if w is None else w[k])
            if ((keys >> np.uint64(32) == mag) & (keys < ref[k])).any():
                return False                  # a partial tie: some element at the cut magnitude is trimmed
    return True


def same_bits(a, b):
    """Bit-identical, NaN payloads aside (a NaN update's payload is not part of the contract)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return bool(((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))).all())


def outside_bracket(d, k_cnt):
    """Full-vector ranks from the cut to a little beyond the sparse sample's rank window: 1.5x (r_lo - rs) of
    ties_sample_ranks, scaled from sample to full ranks (the bracket's bin edges add a few hundred ranks)."""
    nq, s = (d + 3) >> 2, sample_stride(d)
    n_s = d if s == 1 else -(-nq // s) * 8
    rs = k_cnt * n_s / d
    m = 6 * np.sqrt(max(rs * (1 - rs / n_s), 0)) + 8
    return int(1.5 * (np.ceil(rs + m) - rs) * d / n_s)


def magnitude_at(base, m, rank):
    """fp32 |m - b| of the rank-th largest key (1-based)."""
    key = np.partition(keys_of(base, m), base.size - rank)[base.size - rank]
    return np.uint32(key >> np.uint64(32)).view(np.float32)


def density_of(k_cnt, d):
    """A density with int(density * d) == k_cnt (what the oracle's select and the public entry points take)."""
    for x in (k_cnt / d, (k_cnt + 0.5) / d):
        if int(x * d) == k_cnt:
            return x
    raise AssertionError((k_cnt, d))


def block_table(d, G=3):
    """Layer-wise blocks: state-dict-like sizes (a 768 x 768 matrix, biases, an odd-sized tensor), G lambda groups."""
    sizes, ends, grp = [589_824, 768, 3072, 2_359_296, 1_000_003, 777], [], []
    off, i = 0, 0
    while off < d:
        n = min(sizes[i % len(sizes)], d - off)
        if d - off - n < 8:
            n = d - off                      # no block shorter than 8 (the reference's ATen sum changes path there)
        off += n
        ends.append(off)
        grp.append(i % G)
        i += 1
    ends, grp = np.asarray(ends, np.int64), np.asarray(grp, np.int32)
    begins = np.concatenate([[0], ends[:-1]]).astype(np.int64)
    return begins, ends, grp


# ---------------------------------------------------------------------------------------------------- input families
def make_case(family, d, K, seed, k_cnt):
    """(base, models) of one family; the planted families plant into model 0."""
    base, models = synth.make_flat(d, K, seed=seed)
    rng = np.random.default_rng(seed + 7)
    sp = sampled_pairs(d, sample_stride(d))
    ds = sample_stride(d, 4 * SAMPLE_QUADS)
    dp = sampled_pairs(d, ds) if ds >= 4 else np.zeros(0, np.int64)   # stride 2: the dense look reads every quad
    if family in ("high", "high_control"):
        # 500 pairs of the sparse sample (4,000 keys) far above the cut: the sample's order statistic moves about twice
        # the +-(6 sigma + 8) rank window; off the sample, the whole vector's moves by 4,000 ranks, a tenth of the window
        # in sample ranks
        pairs = sp[:: sp.size // 500][:500]
        if family == "high_control":
            pairs = off_sample(pairs, d, [sp, dp])
        cols = pair_columns(pairs, d)
        models[0][cols] = base[cols] + PLANT
    elif family in ("low", "low_control"):
        # 2,500 sampled pairs of model 0 equal to the base (updates of 0): a fifth of their 20,000 keys lay above the cut
        pairs = sp[:: sp.size // 2500][:2500]
        if family == "low_control":
            pairs = off_sample(pairs, d, [sp, dp])
        cols = pair_columns(pairs, d)
        models[0][cols] = base[cols]
    elif family in ("dense", "dense_control"):
        # 2,000 pairs of the dense sample that share no quad with the sparse one: only select_build's third look lies
        only = dp[~np.isin(dp, sp) & ~np.isin(dp + 1, sp) & ~np.isin(dp, sp + 1)]
        pairs = only[:: max(1, only.size // 2000)][:2000]
        if family == "dense_control":
            pairs = off_sample(pairs, d, [sp, dp])
        cols = pair_columns(pairs, d)
        models[0][cols] = base[cols] + PLANT
    elif family.startswith("plateau"):
        # a contiguous run of equal magnitudes (base 0, update +-v) in model 0: 'plateau' puts v at the cut -- the run then
        # fills one final bin and exceeds the final sort; 'plateau_out' puts it just below the bracket; 'plateau_big'
        # puts 100,000 at the cut of a model whose sample lies (the 'high' plants), so that the fast selects fail
        if family == "plateau_big":
            cols = pair_columns(sp[:: sp.size // 500][:500], d)
            models[0][cols] = base[cols] + PLANT
        run = {"plateau": 6000, "plateau_out": 6000, "plateau_big": 100_000}[family]
        v = magnitude_at(base, models[0], k_cnt + (outside_bracket(d, k_cnt) if family == "plateau_out" else 0))
        a = d // 3 + 5
        sign = np.where(rng.random(run) < 0.5, np.float32(-1), np.float32(1))
        base[a:a + run] = 0.0
        for m in models:
            m[a:a + run] = rng.standard_normal(run).astype(np.float32) * np.float32(1e-3)
        models[0][a:a + run] = sign * v
    elif family.startswith("frozen"):
        # 30 % of the columns frozen in 6144-column runs; a tenth of them with base +0 and model -0 (update -0)
        run, n = 6144, int(0.3 * d) // 6144
        starts = rng.choice(d // run, size=n, replace=False) * run
        for i, s in enumerate(starts):
            if i % 10 == 0:
                base[s:s + run] = 0.0
                for m in models:
                    m[s:s + run] = -0.0
            else:
                for m in models:
                    m[s:s + run] = base[s:s + run]
    elif family == "bf16":
        bf = lambda x: torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()  # noqa: E731
        base, models = bf(base), [bf(m) for m in models]
    elif family == "overflow":
        # one element quad out of every 3 * 256 * sm_count -- the thread count of the select's collecting pass (K <= 8) and
        # a multiple of every speculative grid of 1..4 CTAs per SM up to a factor 4: the quads of one or a few threads
        # -- at the cut magnitude.  ~180 keys in the window, but one list of cand_cap (32 at this size) overflows
        period = 3 * 256 * torch.cuda.get_device_properties(0).multi_processor_count
        q = np.arange(0, (d >> 2), period, dtype=np.int64)
        cols = (4 * q[:, None] + np.arange(4)[None, :]).reshape(-1)
        v = magnitude_at(base, models[0], k_cnt)
        base[cols] = 0.0
        models[0][cols] = v
    elif family == "special":
        # NaN (keys above +inf), +-inf, denormal updates, and huge updates that overflow to inf under merge_ties' weights
        idx = rng.choice(d, size=4000, replace=False)
        nan, inf, ninf, den, huge = np.split(idx[:2500], 5)
        models[0][nan] = np.nan
        models[1 % K][inf] = np.inf
        models[0][ninf] = -np.inf
        base[den] = 0.0
        for m in models:
            m[den] = np.float32(3e-39) * np.float32(1 + (den % 7))
        base[huge] = 0.0
        models[K - 1][huge] = np.float32(1e30)
    else:
        assert family == "gauss", family
    return base, models


# ---------------------------------------------------------------------------------------------------- entry points
def deferred_select(tb, tm, k_cnt, w=None):
    cut, status = select_kth_largest(tb, tm, k_cnt, w, defer_status=True)
    return cut_u64(cut).copy(), host(status)


def exact_select(tb, tm, k_cnt, w=None):
    """`mr_ties_select_exact` on its own (the multi-pass path the public entry points fall back to)."""
    lib = _lib.load()
    K, d = len(tm), tb.numel()
    ws_bytes = int(lib.mr_ties_workspace_bytes(d, K))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    cut = torch.zeros(K, dtype=torch.int64, device="cuda")
    status = torch.zeros(K, dtype=torch.int32, device="cuda")
    _lib.check(lib.mr_ties_select_exact(_lib.dptr(tb, torch.float32), _lib.ptr_array(tm), K, d, _lib.dptr(w), int(k_cnt),
                                        _lib.dptr(cut), _lib.dptr(status), _lib.dptr(ws), ws_bytes, _lib.stream_handle()),
               "mr_ties_select_exact")
    assert (host(status) == 1).all(), host(status)
    return cut_u64(cut)


def check_status(tag, status, cut, ref, expect):
    """The central invariant, and the statuses a family is built to produce ({model: status or FAIL}; others: 1)."""
    assert set(status.tolist()) <= STATUSES, (tag, status)
    for k in np.flatnonzero(status == 1):
        assert cut[k] == ref[k], (tag, k, "status 1 with a wrong cut", hex(int(cut[k])), hex(int(ref[k])))
    if expect is None:
        return
    for k in range(status.size):
        want = expect.get(k, DONE)
        if want == FAIL:
            assert status[k] != 1, (tag, k, status)
        else:
            assert status[k] == want, (tag, k, status, want)


def check_case(base, models, k_cnt, tb=None, tm=None, expect_select=None, expect_build=None, weights=None, build=True,
               expect_fused="same"):
    """Every entry point of the select on one input; returns the statuses of the deferred select and select + build."""
    d, K = base.size, len(models)
    if tb is None:
        tb, tm = dev(base), [dev(m) for m in models]
    density = density_of(k_cnt, d)
    ref = ref_cuts(base, models, k_cnt)
    assert np.array_equal(ref, orc.ties_select(base, models, density)), "numpy and C oracle disagree"
    # mr_ties_select, deferred: status 1 => the exact cut; the failures the family is built for
    cut, st = deferred_select(tb, tm, k_cnt)
    check_status("mr_ties_select", st, cut, ref, expect_select)
    # the public select and the exact path: always the cut
    assert np.array_equal(cut_u64(select_kth_largest(tb, tm, k_cnt)), ref), "select_kth_largest"
    assert np.array_equal(exact_select(tb, tm, k_cnt), ref), "mr_ties_select_exact"
    if weights is not None:
        wt = torch.tensor(weights, dtype=torch.float32, device="cuda")
        ref_w = ref_cuts(base, models, k_cnt, weights)
        assert np.array_equal(ref_w, orc.ties_select(base, models, density, weights)), "weighted: numpy and C oracle disagree"
        cut_w, st_w = deferred_select(tb, tm, k_cnt, wt)
        check_status("mr_ties_select weighted", st_w, cut_w, ref_w, None)
        assert np.array_equal(cut_u64(select_kth_largest(tb, tm, k_cnt, wt)), ref_w), "weighted select_kth_largest"
        assert np.array_equal(exact_select(tb, tm, k_cnt, wt), ref_w), "weighted mr_ties_select_exact"
        got = host(merge_ties(tb, tm, list(weights), density))
        assert same_bits(got, orc.merge_ties(base, models, weights, density)), "merge_ties"
    if not build:
        return st, None
    # select + build, deferred, into outputs pre-filled with NaN (unwritten columns show)
    oT = orc.ties_vectors(base, models, density)
    out = alloc_rows(K, d, "cuda")
    out.fill_(float("nan"))
    cut_b, st_b = select_build(tb, tm, k_cnt, _lib.MR_TIES_VECTORS, out, ldo=max(out.stride(0), d), defer_status=True)
    cut_b, st_b = cut_u64(cut_b), host(st_b)
    check_status("select_build VECTORS", st_b, cut_b, ref, expect_build)
    if (st_b == 1).all():
        assert same_bits(host(out), oT), "select_build VECTORS output, status 1"
    rng = np.random.default_rng(d % 9973)
    sb, se, sg = block_table(d)
    for layer_wise in (False, True):
        G = 3 if layer_wise else 1
        w = rng.uniform(0.1, 0.6, size=(G, K)).astype(np.float32)
        want = orc.lambda_merge(base, oT, w, sb, se, sg) if layer_wise else orc.lambda_merge(base, oT, w)
        seg_end, seg_group = (dev(se), dev(sg)) if layer_wise else (None, None)
        fused = torch.full((d,), float("nan"), device="cuda")
        cut_f, st_f = select_build(tb, tm, k_cnt, _lib.MR_TIES_FUSED_MERGE, fused, w=dev(w), G=G, seg_end=seg_end,
                                   seg_group=seg_group, defer_status=True)
        st_f = host(st_f)
        check_status(f"select_build FUSED_MERGE layer_wise={layer_wise}", st_f, cut_u64(cut_f), ref,
                     expect_build if expect_fused == "same" else expect_fused)
        if (st_f == 1).all():
            assert same_bits(host(fused), want), ("FUSED_MERGE output, status 1", layer_wise)
        # the public one-pass merge: exact whatever the sample said
        got = host(merge_ties_lambda(tb, tm, density, dev(w), seg_end, seg_group))
        assert same_bits(got, want), ("merge_ties_lambda", layer_wise)
    assert same_bits(host(get_ties_vectors(tb, tm, density)), oT), "get_ties_vectors"
    return st, st_b


# ---------------------------------------------------------------------------------------------------- the families
D5, D20, D3 = 5_000_017, 20_000_003, 3_000_017
# Regression cases (test_sample_lies[low-3 M], test_dense_sample_lies[dense]): a sample pick that clamps a rank above
# the bracket used to make a bracket starting above its own end; that model's full pass then collected almost every key,
# and mr_ties_select_build reported 1 with a wrong cut for the model next to it.


def test_mirror_makes_strict_subsamples():
    """The sizes used below: both samples are strict subsamples (stride >= 4 quads), except the sparse-only 3 M case."""
    for d in (D5, D20):
        assert sample_stride(d) >= 4 and sample_stride(d, 4 * SAMPLE_QUADS) >= 4, d
    assert sample_stride(D3) >= 4 and sample_stride(D3, 4 * SAMPLE_QUADS) == 2
    assert (sample_stride(D20), sample_stride(D20, 4 * SAMPLE_QUADS)) == (76, 18)


@pytest.mark.parametrize("d,K,density", [(D5, 1, 0.2), (D5, 5, 0.01), (D5, 8, 0.99), (D3, 16, 0.5), (D20, 2, 0.2)],
                         ids=lambda x: str(x))
def test_control_gaussian(d, K, density):
    """Gaussian updates: every model's sample tells the truth, every entry point reports 1 and the exact cut."""
    base, models = synth.make_flat(d, K, seed=d % 101 + K)
    k_cnt = int(density * d)
    weights = [0.7, -1.3, 0.0, 2.0, 0.5][:K] + [0.3] * max(0, K - 5) if K > 1 else None
    check_case(base, models, k_cnt, expect_select={}, expect_build={}, weights=weights)


@pytest.mark.parametrize("d,K", [(D5, 3), (D20, 2), (D3, 2)], ids=lambda x: str(x))
@pytest.mark.parametrize("family,expect", [("high", BRACKET_HIGH), ("high_control", DONE),
                                           ("low", BRACKET_LOW), ("low_control", DONE)])
def test_sample_lies(family, expect, d, K):
    """Plants at exactly the sparse-sampled quads of model 0.  Large updates make the sample put the bracket ABOVE the
    cut (the target lies below it: TIES_ERR_BRACKET_HIGH); updates of 0 put it below (more than k_cnt - 1 keys above it:
    TIES_ERR_BRACKET_LOW).  The controls move every plant one pair off both samples and must report 1."""
    k_cnt = int(0.2 * d)
    base, models = make_case(family, d, K, seed=11, k_cnt=k_cnt)
    check_case(base, models, k_cnt, expect_select={0: expect}, expect_build={0: expect}, build=d != D20)


@pytest.mark.parametrize("family", ["high", "plateau"])
@pytest.mark.parametrize("shift", [1, 3])
def test_unaligned_pointers(family, shift):
    """The scalar-load instantiations on the families that must fail."""
    d, K = D5, 2
    k_cnt = int(0.2 * d)
    base, models = make_case(family, d, K, seed=23, k_cnt=k_cnt)
    tb, tm = shifted(base, shift, d), [shifted(m, shift, d) for m in models]
    code = BRACKET_HIGH if family == "high" else TOO_MANY
    check_case(base, models, k_cnt, tb, tm, expect_select={0: code}, expect_build={0: code})


@pytest.mark.parametrize("family", ["dense", "dense_control"])
def test_dense_sample_lies(family):
    """Plants at quads that only the dense (third) sample of `mr_ties_select_build` picks: its bracket misses and it must
    say so; `mr_ties_select` never looks there and reports 1."""
    d, K = D20, 2
    k_cnt = int(0.2 * d)
    base, models = make_case(family, d, K, seed=31, k_cnt=k_cnt)
    check_case(base, models, k_cnt, expect_select={}, expect_build={0: BRACKET_HIGH} if family == "dense" else {})


@pytest.mark.parametrize("family,expect", [("plateau", TOO_MANY), ("plateau_out", DONE)])
def test_plateau_at_the_cut(family, expect):
    """6,000 equal magnitudes in consecutive columns, at the cut: the bracket spans many magnitudes, so the two 1024-way
    refinements leave the whole run in one bin and the final sort cannot take it (TIES_ERR_TOO_MANY).  The same run
    just below the sample's rank window (1.5x its half-width below the cut) lies outside the bracket and must resolve."""
    d, K = D5, 3
    k_cnt = int(0.2 * d)
    base, models = make_case(family, d, K, seed=41, k_cnt=k_cnt)
    check_case(base, models, k_cnt, expect_select={0: expect}, expect_build={0: expect})


# Regression case (density 0.99): the cut inside the frozen zeros makes the speculative pass collect every +-0 element,
# which slows its warps enough that a stage of its shared-memory ring was refilled before every warp had read it (the
# refill, an async-proxy write, was not ordered after the generic reads): some columns came out of other columns' data
# with every status 1.
@pytest.mark.parametrize("density", [0.8, 0.99, 0.2])
def test_frozen_columns(density):
    """30 % of the columns frozen in tensor-sized runs (updates +0, and -0 where base is +0 and the model -0): at
    densities 0.8 and 0.99 the cut lies inside the zeros and is decided by the lowest-index rule across +0 and -0."""
    d, K = D5, 3
    k_cnt = int(density * d)
    base, models = make_case("frozen", d, K, seed=51, k_cnt=k_cnt)
    check_case(base, models, k_cnt, weights=[0.5, -2.0, 1.0])


def test_bf16_rounded_checkpoints():
    d, K = D5, 4
    k_cnt = int(0.2 * d)
    base, models = make_case("bf16", d, K, seed=61, k_cnt=k_cnt)
    check_case(base, models, k_cnt, weights=[0.25, 0.5, -0.75, 1.0])


def test_one_candidate_list_overflows():
    """~180 in-window keys on the quads of one thread of the collecting grid: few keys in the window overall, but one
    list exceeds cand_cap.  The select must report TIES_ERR_CAND_OVERFLOW, select + build (VECTORS, grid-stride tiles)
    a failure; FUSED_MERGE hands each CTA a contiguous range of tiles, so the planted quads land in different lists and
    only the invariant applies there."""
    d, K = D20, 2
    k_cnt = int(0.2 * d)
    base, models = make_case("overflow", d, K, seed=71, k_cnt=k_cnt)
    check_case(base, models, k_cnt, expect_select={0: CAND_OVERFLOW}, expect_build={0: FAIL}, expect_fused=None)


def test_special_values():
    """NaN updates (keys above +inf), +-inf, denormals, and w * u overflowing to inf in merge_ties."""
    d, K = D5, 3
    k_cnt = int(0.2 * d)
    base, models = make_case("special", d, K, seed=81, k_cnt=k_cnt)
    check_case(base, models, k_cnt, weights=[1.0, 0.5, 1e10])


# ---------------------------------------------------------------------------------------------------- sharded
@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("planted", [False, True])
def test_dist_select_shards_with_different_statistics(world, planted):
    """`DistSelect` over emulated ranks: rank 0's slice frozen in every model; with `planted`, model 0's updates at the
    sparse-sampled quads of the last rank's slice (every rank samples its slice with the global stride from its own
    quad 0).  All ranks report the same status; status 1 means the global cut is the reference and the local cuts
    rebuild each slice of the oracle's vectors bit for bit; the planted model must fail."""
    d, K = D5, 3
    k_cnt = int(0.2 * d)
    base, models = synth.make_flat(d, K, seed=90 + world)
    lo0, hi0 = flat_shard_bounds(d, world, 0)
    for m in models:
        m[lo0:hi0] = base[lo0:hi0]
    if planted:
        lo, hi = flat_shard_bounds(d, world, world - 1)
        cols = lo + pair_columns(sampled_pairs(hi - lo, sample_stride(d))[::10], hi - lo)
        models[0][cols] = base[cols] + PLANT
    ref = ref_cuts(base, models, k_cnt)
    fb, fm = dev(base), [dev(m) for m in models]
    sels = _emulated_dist_select(fb, fm, k_cnt, world)
    statuses = [host(s.status) for s in sels]
    assert all(np.array_equal(s, statuses[0]) for s in statuses), statuses
    st = statuses[0]
    check_status("DistSelect", st, cut_u64(sels[0].cut_global), ref, {0: FAIL} if planted else {})
    for s in sels:
        assert np.array_equal(cut_u64(s.cut_global)[st == 1], ref[st == 1])
    if (st == 1).all():
        from mergerec_b200.merger.algorithms.ties import _build
        oT = orc.ties_vectors(base, models, density_of(k_cnt, d))
        for r, s in enumerate(sels):
            lo, hi = flat_shard_bounds(d, world, r)
            part = alloc_rows(K, hi - lo, "cuda")
            _build(s.base, s.rows, s.cut, _lib.MR_TIES_VECTORS, out=part, ldo=max(part.stride(0), hi - lo))
            assert np.array_equal(host(part).view(np.uint32), oT[:, lo:hi].view(np.uint32)), r
    # the public sharded select at world 1 on the same input
    assert same_survivors(base, models, cut_u64(sharded_select(fb, fm, k_cnt, d)), ref)


@pytest.mark.parametrize("family", ["high", "low", "dense", "plateau", "plateau_big", "frozen", "overflow", "special"])
def test_sharded_select_world1(family):
    """`sharded_select` (world 1, non-deferred) keeps exactly the reference's survivors on every family; 'plateau_big' (100,000 equal
    magnitudes straddling the cut, more than the 65,536-entry tie list) makes the exact windowed search rescan the slice
    for the tied index."""
    d, K = (D20, 2) if family in ("dense", "overflow") else (D5, 3)
    k_cnt = int(0.2 * d)
    base, models = make_case(family, d, K, seed=101, k_cnt=k_cnt)
    fb, fm = dev(base), [dev(m) for m in models]
    assert same_survivors(base, models, cut_u64(sharded_select(fb, fm, k_cnt, d)), ref_cuts(base, models, k_cnt)), family
    if family == "plateau_big":
        _, st = deferred_select(fb, fm, k_cnt)
        assert st[0] != 1, st
