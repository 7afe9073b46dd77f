"""GPU parity for TIES (A6-A9): CUDA select + build kernels through the C ABI against the reference's golden
vectors and the CPU oracle.  Masks, cut keys and vectors are compared bit-for-bit under the canonical
lowest-index tie rule; against the raw reference (torch.topk's unspecified tie order) differences must be
confined to columns holding a threshold-magnitude entry."""
import numpy as np
import pytest
import torch

import golden_cases as gc
from helpers import assert_bit_equal, golden
from mergerec_b200 import synth
from mergerec_b200.merger.algorithms import get_ties_vectors, merge_ties
from mergerec_b200.merger.algorithms.ties import merge_ties_lambda, ties_select, ties_topk_count
from mergerec_b200.merger.layout import FlatLayout
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().cpu().numpy()


def cut_u64(t):
    return host(t).view(np.uint64)


def check_against_oracle(base, models, density, weights=None):
    tb, tm = dev(base), [dev(m) for m in models]
    That, trim, elect, cut = get_ties_vectors(tb, tm, density, return_masks=True)
    oT, otrim, oelect, ocut = orc.ties_vectors(base, models, density, return_masks=True)
    assert np.array_equal(cut_u64(cut), ocut), "cut keys"
    assert np.array_equal(host(trim), otrim), "trim mask"
    assert np.array_equal(host(elect), oelect), "elect mask"
    assert_bit_equal(host(That), oT, "TIES vectors")
    if weights is not None:
        assert_bit_equal(host(merge_ties(tb, tm, weights, density)), orc.merge_ties(base, models, weights, density),
                         "merge_ties")
    return That, cut


@pytest.mark.parametrize("case", gc.TIES_CASES, ids=lambda c: c["name"])
def test_ties_vs_golden_and_oracle(case):
    g = golden("ties")
    base, models = synth.make_flat(case["d"], case["K"], seed=case["seed"], tie_free=case["tie_free"],
                                   quantize=case.get("quantize", 0.0))
    That, cut = check_against_oracle(base, models, case["density"], case["weights"])
    ref_T = g[f"{case['name']}/ties_vectors"]
    ref_M = g[f"{case['name']}/merge_ties"]
    tb, tm = dev(base), [dev(m) for m in models]
    if case["tie_free"]:
        assert_bit_equal(host(That), ref_T, "get_ties_vectors vs raw reference")
        assert_bit_equal(host(merge_ties(tb, tm, case["weights"], case["density"])), ref_M, "merge_ties vs raw reference")
    else:
        thr = (cut_u64(cut) >> np.uint64(32)).astype(np.uint32)
        diff_cols = (host(That).view(np.uint32) != ref_T.view(np.uint32)).any(axis=0)
        col_has_thr = np.zeros(case["d"], bool)
        for k, m in enumerate(models):
            col_has_thr |= np.abs(m - base).view(np.uint32) == thr[k]
        assert not (diff_cols & ~col_has_thr).any(), "difference vs raw torch.topk outside threshold ties"


def test_ties_edge_densities_and_all_ties():
    base, models = synth.make_flat(1000, 3, seed=5)
    tb, tm = dev(base), [dev(m) for m in models]
    for density, expect in [(0.0, 0), (1.0, 1000), (0.0004, 0), (0.9999, 999), (0.001, 1)]:
        _, trim, _, _ = get_ties_vectors(tb, tm, density, return_masks=True)
        assert (host(trim).sum(axis=1) == expect).all(), density
    # a model identical to the base: every |u| == 0 -> all ties -> the lowest indices survive (exact fallback path)
    check_against_oracle(base, [base.copy(), models[0]], 0.25)
    _, trim, _, _ = get_ties_vectors(tb, [tb.clone(), tm[0]], 0.25, return_masks=True)
    trim = host(trim)
    assert trim[0, :250].all() and not trim[0, 250:].any()


@pytest.mark.parametrize("K", [1, 2, 5, 9, 16])
def test_ties_all_k(K):
    d = 32 * 97 + 7
    base, models = synth.make_flat(d, K, seed=300 + K)
    w = [0.2 + 0.05 * k for k in range(K)]
    check_against_oracle(base, models, 0.3, w)


@pytest.mark.parametrize("shift", [1, 2])
def test_ties_unaligned(shift):
    K, d = 4, 6001
    base, models = synth.make_flat(d + 4, K, seed=88)
    tb = dev(base)[shift:shift + d]
    tm = [dev(m)[shift:shift + d] for m in models]
    hb, hm = base[shift:shift + d], [m[shift:shift + d] for m in models]
    That = get_ties_vectors(tb, tm, 0.2)
    assert_bit_equal(host(That), orc.ties_vectors(hb, hm, 0.2), "unaligned TIES vectors")
    w = [0.5, 0.25, 1.0, 0.75]
    assert_bit_equal(host(merge_ties(tb, tm, w, 0.2)), orc.merge_ties(hb, hm, w, 0.2), "unaligned merge_ties")


def test_ties_heavy_ties_quantised():
    """Quantised updates: thousands of equal magnitudes at the threshold; the tie cut must be by lowest index."""
    K, d = 3, 200_003
    base, models = synth.make_flat(d, K, seed=9, quantize=5e-4)
    check_against_oracle(base, models, 0.2, [0.3, 0.3, 0.3])


def test_ties_sampled_path_medium():
    """d large enough that the sample stride is > 1 (the bracket comes from a strict subsample)."""
    K, d = 4, 3_000_017
    base, models = synth.make_flat(d, K, seed=12)
    tb, tm = dev(base), [dev(m) for m in models]
    cut = ties_select(tb, tm, 0.2)
    assert np.array_equal(cut_u64(cut), orc.ties_select(base, models, 0.2))
    w = torch.tensor([0.3, -0.4, 0.5, 0.0], dtype=torch.float32, device="cuda")  # w = 0 -> all-zero updates -> all ties
    cutw = ties_select(tb, tm, 0.2, w)
    assert np.array_equal(cut_u64(cutw), orc.ties_select(base, models, 0.2, [0.3, -0.4, 0.5, 0.0]))


@pytest.mark.parametrize("recformer", [False, True])
@pytest.mark.parametrize("layer_wise", [False, True])
def test_fused_ties_lambda_merge(recformer, layer_wise):
    """merge_ties_lambda == get_ties_vectors followed by the lambda merge (bit-exact, incl. ragged blocks)."""
    K = 6
    shapes = synth.tiny_shapes(recformer=recformer)
    sbase, smodels = synth.make_state_dicts(shapes, K, seed=70, sigma=1e-2)
    base = np.concatenate([np.asarray(v).reshape(-1).astype(np.float32) for v in sbase.values()])
    models = [np.concatenate([np.asarray(v).reshape(-1).astype(np.float32) for v in m.values()]) for m in smodels]
    sb, se, sg, keys = orc.segment_table(shapes, layer_wise=layer_wise)
    rng = np.random.Generator(np.random.PCG64(3))
    w = rng.uniform(0.1, 0.6, size=(len(keys), K)).astype(np.float32)
    want = orc.lambda_merge(base, orc.ties_vectors(base, models, 0.2), w, sb, se, sg)
    layout = FlatLayout.from_shape_dict(shapes)
    seg_end, seg_group, _ = layout.device_blocks(layer_wise, "cuda")
    got = merge_ties_lambda(dev(base), [dev(m) for m in models], 0.2, dev(w),
                            seg_end if layer_wise else None, seg_group if layer_wise else None)
    assert_bit_equal(host(got), want, "fused TIES + lambda merge")


def test_ties_full_size_blair_base():
    """BASELINE config 2 size: K = 8, d = 124,645,632, density 0.2; cut keys and TIES vectors bit-exact vs the oracle."""
    d, K = synth.total_numel(synth.roberta_shapes()), 8
    g = torch.Generator(device="cuda").manual_seed(6)
    base = torch.randn(d, generator=g, device="cuda") * 0.02
    models = [base + 1e-3 * torch.randn(d, generator=g, device="cuda") for _ in range(K)]
    That, trim, elect, cut = get_ties_vectors(base, models, 0.2, return_masks=True)
    k_cnt = ties_topk_count(0.2, d)
    assert k_cnt == 24_929_126
    assert (trim.sum(dim=1) == k_cnt).all(), "every model keeps exactly int(density*d) entries"
    assert torch.equal(elect, That != 0)
    hb, hm = host(base), [host(m) for m in models]
    assert np.array_equal(cut_u64(cut), orc.ties_select(hb, hm, 0.2))
    want = orc.ties_vectors(hb, hm, 0.2)
    got = host(That)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("case", gc.LNS_CASES, ids=lambda c: c["name"])
def test_localize_and_stitch_vs_golden_and_oracle(case):
    """SURVEY.md section 8(f) row 2: Localize-and-Stitch vectors and merge through the TIES select + build kernels."""
    from mergerec_b200.merger.algorithms import get_localize_and_stitch_vectors, merge_localize_and_stitch
    g = golden("lns")
    base, models = synth.make_flat(case["d"], case["K"], seed=case["seed"], tie_free=case["tie_free"])
    tb, tm = dev(base), [dev(m) for m in models]
    vec = host(get_localize_and_stitch_vectors(tb, tm, case["density"]))
    merged = host(merge_localize_and_stitch(tb, tm, case["weights"], case["density"]))
    assert_bit_equal(vec, orc.lns_vectors(base, models, case["density"]), "L&S vectors vs oracle")
    assert_bit_equal(merged, orc.merge_localize_and_stitch(base, models, case["weights"], case["density"]), "L&S merge")
    if case["tie_free"]:
        assert_bit_equal(vec, g[f"{case['name']}/vectors"], "L&S vectors vs raw reference")
        assert_bit_equal(merged, g[f"{case['name']}/merged"], "L&S merge vs raw reference")


def test_localize_and_stitch_module(monkeypatch):
    """load_merging_module(MergeType.LOCALIZE_AND_STITCH, ...) builds the stitched vectors and merges them."""
    from toy_model import ToyEncoder, make_toy_state_dicts
    from mergerec_b200.merger.enums import LearnType, MergeType
    from mergerec_b200.merger.weight_learning.module import load_merging_module
    pre, fts = make_toy_state_dicts(4, seed=81)
    torch.manual_seed(1)
    mod = load_merging_module(MergeType.LOCALIZE_AND_STITCH, LearnType.TASK_WISE, ToyEncoder(), pre, fts, ignore_keys=set(),
                              ties_density=0.1, initial_per_weight=1.0, disable_softmax=True)
    keys = list(pre.keys())
    fb = np.concatenate([pre[k].numpy().reshape(-1).astype(np.float32) for k in keys])
    fm = [np.concatenate([ft[k].numpy().reshape(-1).astype(np.float32) for k in keys]) for ft in fts]
    want = orc.merge_localize_and_stitch(fb, fm, [1.0] * 4, 0.1)
    sd = mod.get_state_dict()
    got = np.concatenate([sd[k].detach().cpu().numpy().reshape(-1) for k in keys])
    assert_bit_equal(got, want, "merged state_dict through the L&S module")


# ------------------------------------------------------------------------------------------ one-pass select + build
def _spec_case(K, d, seed, quantize=0.0, density=0.2, shift=0):
    from mergerec_b200 import _lib
    from mergerec_b200.merger.algorithms.ties import _build, select_build, select_kth_largest
    from mergerec_b200.merger.layout import alloc_rows
    base, models = synth.make_flat(d, K, seed=seed, quantize=quantize)
    if shift:      # pointers off the 16-byte grid: the scalar-load instantiation
        buf = torch.empty((K + 1) * (d + 8) + 8, dtype=torch.float32, device="cuda")
        views = [buf[i * (d + 8) + shift: i * (d + 8) + shift + d] for i in range(K + 1)]
        views[0].copy_(dev(base))
        for v, m in zip(views[1:], models):
            v.copy_(dev(m))
        tb, tm = views[0], views[1:]
    else:
        tb, tm = dev(base), [dev(m) for m in models]
    k_cnt = ties_topk_count(density, d)
    cut = select_kth_largest(tb, tm, k_cnt)
    want = alloc_rows(K, d, "cuda")
    _build(tb, tm, cut, _lib.MR_TIES_VECTORS, out=want, ldo=max(want.stride(0), d))
    got = alloc_rows(K, d, "cuda")
    got.fill_(float("nan"))
    cut2, status = select_build(tb, tm, k_cnt, _lib.MR_TIES_VECTORS, got, ldo=max(got.stride(0), d), defer_status=True)
    return tb, tm, k_cnt, cut, want, got, cut2, status


@pytest.mark.parametrize("K,d,quantize", [(1, 4096, 0.0), (2, 100_003, 0.0), (3, 262_144 + 17, 0.0), (5, 300_031, 0.0),
                                          (8, 1_000_003, 0.0), (8, 524_288, 2.5e-4), (16, 200_001, 0.0), (4, 37, 0.0),
                                          (7, 2_000_029, 1e-5)])
def test_select_build_equals_select_then_build(K, d, quantize):
    """`mr_ties_select_build` (speculative build + exact cut + fix-up) == `mr_ties_select` + `mr_ties_build`, bit for bit:
    cut keys and every element of the (K, d) TIES vectors, including the interleaved-order tail columns (K >= 5), a partial
    last quad, and inputs with many equal magnitudes around the cut."""
    tb, tm, k_cnt, cut, want, got, cut2, status = _spec_case(K, d, seed=300 + K, quantize=quantize)
    _check_deferred_status(tb, tm, k_cnt, cut, want, got, cut2, status)
    # thousands of equal magnitudes at the cut (quantised inputs) may defeat the two 1024-way refinements; nothing else may
    assert status.cpu().tolist() == [1] * K or quantize > 0, status.cpu().tolist()


def _check_deferred_status(tb, tm, k_cnt, cut, want, got, cut2, status):
    """A deferred select + build: every model reporting 1 carries the exact cut, a failure is one of the TIES_ERR_*
    codes, all 1 means the output is exact, and the public (non-deferred) call is exact whatever the status."""
    from mergerec_b200 import _lib
    from mergerec_b200.merger.algorithms.ties import select_build
    from mergerec_b200.merger.layout import alloc_rows
    st = status.cpu()
    assert set(st.tolist()) <= {1, -1, -2, -3, -4, -5}, st.tolist()
    assert torch.equal(cut2.cpu()[st == 1], cut.cpu()[st == 1]), "status 1 with a wrong cut"
    if bool((st == 1).all()):
        assert torch.equal(cut2, cut)
        assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    K, d = len(tm), tb.numel()
    pub = alloc_rows(K, d, "cuda")
    pub.fill_(float("nan"))
    assert torch.equal(select_build(tb, tm, k_cnt, _lib.MR_TIES_VECTORS, pub, ldo=max(pub.stride(0), d)), cut)
    assert torch.equal(pub.view(torch.int32), want.view(torch.int32))


@pytest.mark.parametrize("shift", [1, 2, 3])
def test_select_build_unaligned_pointers(shift):
    _, _, _, cut, want, got, cut2, status = _spec_case(8, 150_001, seed=77, shift=shift)
    assert status.cpu().tolist() == [1] * 8
    assert torch.equal(cut2, cut) and torch.equal(got.view(torch.int32), want.view(torch.int32))


@pytest.mark.parametrize("density", [0.0, 1e-7, 0.01, 0.5, 0.999, 1.0])
def test_select_build_edge_densities(density):
    tb, tm, k_cnt, cut, want, got, cut2, status = _spec_case(5, 70_001, seed=5, density=density)
    _check_deferred_status(tb, tm, k_cnt, cut, want, got, cut2, status)


def test_select_build_falls_back_on_massive_ties():
    """All updates equal in magnitude: the sampled bracket cannot isolate the cut; the public entry points must notice and
    still return the exact answer (exact select + plain build)."""
    d, K = 300_000, 3
    base = np.zeros(d, np.float32)
    models = [np.full(d, 0.5, np.float32) * (1 if k % 2 == 0 else -1) for k in range(K)]
    got = get_ties_vectors(dev(base), [dev(m) for m in models], 0.2)
    want = orc.ties_vectors(base, models, 0.2)
    assert_bit_equal(host(got)[:, :d], want, "massive ties")


@pytest.mark.parametrize("recformer,K", [(False, 3), (True, 8), (False, 5)])
def test_fused_select_build_merge_layerwise(recformer, K):
    """FUSED_MERGE through the one-pass kernel: layer-wise lambdas over a state_dict-shaped block table (blocks that
    straddle quads, blocks shorter than a quad, per-block interleaved tails) == materialised T-hat + lambda merge."""
    from mergerec_b200 import _lib
    from mergerec_b200.merger.algorithms._common import merge_axpy
    shapes = synth.tiny_shapes(layers=3, hidden=40, ffn=72, vocab=301, max_pos=18, recformer=recformer)
    layout = FlatLayout.from_shape_dict(shapes)
    d = layout.d
    base, models = synth.make_flat(d, K, seed=900 + K)
    tb, tm = dev(base), [dev(m) for m in models]
    seg_end, seg_group, keys = layout.device_blocks(True, tb.device)
    rng = np.random.Generator(np.random.PCG64(3))
    w = dev(rng.uniform(0.1, 0.5, size=(len(keys), K)).astype(np.float32))
    That = get_ties_vectors(tb, tm, 0.2)
    two_step = merge_axpy(tb, list(That.unbind(0)), w, _lib.MR_ORDER_SUM_FIRST, False, seg_end, seg_group)
    fused = merge_ties_lambda(tb, tm, 0.2, w, seg_end, seg_group, one_pass=True)
    assert torch.equal(fused.view(torch.int32), two_step.view(torch.int32))
    assert torch.equal(merge_ties_lambda(tb, tm, 0.2, w, seg_end, seg_group).view(torch.int32), two_step.view(torch.int32))
    cut = ties_select(tb, tm, 0.2)
    fused_given_cut = merge_ties_lambda(tb, tm, 0.2, w, seg_end, seg_group, cut=cut)
    assert torch.equal(fused_given_cut.view(torch.int32), two_step.view(torch.int32))
    # task-wise lambdas (one block)
    w1 = dev(rng.uniform(0.1, 0.5, size=(1, K)).astype(np.float32))
    two_step1 = merge_axpy(tb, list(That.unbind(0)), w1, _lib.MR_ORDER_SUM_FIRST, False)
    assert torch.equal(merge_ties_lambda(tb, tm, 0.2, w1, one_pass=True).view(torch.int32), two_step1.view(torch.int32))
    assert torch.equal(merge_ties_lambda(tb, tm, 0.2, w1).view(torch.int32), two_step1.view(torch.int32))
    oT = orc.ties_vectors(base, models, 0.2)
    assert_bit_equal(host(That)[:, :d], oT, "one-pass TIES vectors vs oracle")
