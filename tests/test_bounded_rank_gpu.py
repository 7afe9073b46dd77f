"""GPU: label ranks bounded by a cap (`Evaluator.label_ranks(cap=...)`, `bounded_count`) -- a probe over a slice of the
catalog, the live rows compacted (`mr_rank_compact`, `mr_rank_gather`), the rest counted for them alone and added
(`mr_rank_add`) -- and `evaluate_embeddings`, which ranks with cap = max(ks).

Exact bar: a bounded rank equals the exact rank (`label_ranks()`) wherever that is below the cap and is >= the cap
elsewhere; a query's count does not depend on the row it lands in after compaction; the metric floats equal those of
the top-K lists bit for bit."""
import numpy as np
import pytest
import torch

from mergerec_b200 import synth
from mergerec_b200.evaluator import Evaluator, ShardedItemTable, shard_bounds
from mergerec_b200.evaluator import evaluator as evm
from mergerec_b200.evaluator.evaluator import exclusion_csr, label_score, score_rank
from mergerec_b200.evaluator.sharded import MR_SCORE_BF16, MR_SCORE_TF32X1, MR_SCORE_TF32X3
from oracle import oracle as orc
from test_exclude_gpu import big_gauss, make_histories
from test_label_rank_gpu import GRID_SHAPES, make_labels

pytestmark = pytest.mark.gpu

ID_BASE = 1000
MODES = (MR_SCORE_TF32X3, MR_SCORE_TF32X1, MR_SCORE_BF16)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def assert_bounded(got, exact, cap, what=""):
    got, exact = got.cpu().numpy(), exact.cpu().numpy()
    assert got.dtype == np.int32
    below = (exact >= 0) & (exact < cap)
    assert np.array_equal(got[below], exact[below]), f"exact part, {what}"
    assert np.array_equal(got < 0, exact < 0), f"misses, {what}"
    assert (got[exact >= cap] >= cap).all(), f"bounded part, {what}"


def assert_same_count_anywhere(q, table, tl, key, mode, exclude, sel):
    """score_rank of the queries `sel` (any order), gathered into rows of their own, against their in-place counts."""
    Q = tl.shape[0]
    csr = None if exclude is None else exclusion_csr(exclude, Q)
    full = score_rank(q.hi, q.lo, table, tl, key, mode, csr)
    csr_s = None if exclude is None else exclusion_csr(exclude[sel], sel.numel())
    lo = None if q.lo is None else q.lo[sel].contiguous()
    got = score_rank(q.hi[sel].contiguous(), lo, table, tl[sel].contiguous(), key[sel].contiguous(), mode, csr_s)
    assert torch.equal(got, full[sel]), f"mode {mode}, exclude {exclude is not None}"


def subsets(Q, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    half = torch.nonzero(torch.rand(Q, generator=g, device="cuda") < 0.5).flatten()     # ascending, as compacted
    return half, torch.randperm(Q, generator=g, device="cuda")[: max(1, Q // 3)]        # and shuffled


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("shape", GRID_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_counts_do_not_depend_on_the_query_row_grid(shape, cg, monkeypatch):
    monkeypatch.setenv("MR_SCORE_CTA_GROUP", str(cg))
    Q, N, E = shape
    users, items, _ = synth.make_catalog(Q, N, E, kind="grid", seed=211)
    scores = orc.scores_f32(users, items)
    labels = make_labels(scores, ID_BASE, seed=212)
    ex = dev(make_histories(scores, 20, labels, ID_BASE, seed=213))
    ev = Evaluator(["RECALL"], [10])
    tl = dev(labels)
    for mode in MODES:
        if mode == MR_SCORE_BF16 and E % 8:
            continue
        table = ShardedItemTable(dev(items), id_base=ID_BASE, bf16=mode == MR_SCORE_BF16)
        q = ev.prepare_queries(dev(users), mode=mode)
        key = label_score(q.hi, q.lo, table, tl, mode)
        for sel in subsets(Q, 214):
            for exclude in (None, ex):
                assert_same_count_anywhere(q, table, tl, key, mode, exclude, sel)


@pytest.mark.parametrize("cg", [1, 2])
def test_counts_do_not_depend_on_the_query_row_at_scale(cg, monkeypatch):
    """Gaussian 4,096 x 1,000,000 x 768: the counts of compacted queries are the counts in place, bit for bit."""
    monkeypatch.setenv("MR_SCORE_CTA_GROUP", str(cg))
    Q, N, E = 4096, 1_000_000, 768
    users, items = big_gauss(Q, N, E, seed=221)
    g = torch.Generator(device="cuda").manual_seed(222)
    tl = torch.randint(0, N, (Q,), generator=g, device="cuda")
    ex = torch.randint(-1, N, (Q, 50), generator=g, device="cuda")
    ev = Evaluator(["RECALL"], [10])
    for mode in MODES:
        table = ShardedItemTable(items, bf16=mode == MR_SCORE_BF16)
        q = ev.prepare_queries(users, mode=mode)
        key = label_score(q.hi, q.lo, table, tl, mode)
        for sel in subsets(Q, 223):
            for exclude in (None, ex):
                assert_same_count_anywhere(q, table, tl, key, mode, exclude, sel)
        del table, q


@pytest.mark.parametrize("max_live", [0.0, 0.9, 1.0], ids=["in_place", "default", "always_compact"])
@pytest.mark.parametrize("shape", GRID_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_bounded_ranks_grid(shape, max_live, monkeypatch):
    """make_labels' cases (outside the table, tied, last partial tile), exclusion lists, probes of 1 .. 4 tiles and of
    the whole table, caps from 1 to past N (Q_live = Q), both sides of the skip rule."""
    monkeypatch.setattr(evm, "COMPACT_MAX_LIVE", max_live)
    Q, N, E = shape
    users, items, _ = synth.make_catalog(Q, N, E, kind="grid", seed=231)
    scores = orc.scores_f32(users, items)
    labels = make_labels(scores, ID_BASE, seed=232)
    ex = dev(make_histories(scores, 20, labels, ID_BASE, seed=233))
    ev = Evaluator(["RECALL"], [10])
    tl = dev(labels)
    for mode in MODES:
        if mode == MR_SCORE_BF16 and E % 8:
            continue
        table = ShardedItemTable(dev(items), id_base=ID_BASE, bf16=mode == MR_SCORE_BF16)
        q = ev.prepare_queries(dev(users), mode=mode)
        for exclude in (None, ex):
            exact = ev.label_ranks(q, table, tl, mode=mode, exclude=exclude)
            for div in ("1", "3", "64", "100000"):
                monkeypatch.setenv("MR_SCORE_PROBE_DIV", div)
                for cap in (1, 10, 100, N + 1):
                    got = ev.label_ranks(q, table, tl, mode=mode, exclude=exclude, cap=cap)
                    assert_bounded(got, exact, cap, f"mode {mode} div {div} cap {cap}")


def test_bounded_ranks_special_values_and_edges(monkeypatch):
    """NaN and +-0 scores, ids that end at 2^31 - 1, no live row (no label in the table), every row live."""
    Q, N, E = 300, 2000, 64
    rng = np.random.Generator(np.random.PCG64(241))
    users = rng.integers(-2, 3, (Q, E)).astype(np.float32)
    items = rng.integers(-2, 3, (N, E)).astype(np.float32)
    items[rng.random(N) < 0.05] = 0.0
    items[rng.random(N) < 0.02, 0] = np.nan
    users[::11] = 0.0
    users[5::11, :E // 2] = -0.0
    ev = Evaluator(["RECALL"], [10])
    for id_base in (ID_BASE, 2 ** 31 - 1 - N):
        labels = rng.integers(0, N, Q) + id_base
        labels[::13] = id_base + np.argmax(np.isnan(items[:, 0]))
        outside = np.full(Q, id_base - 1)
        for mode in MODES:
            table = ShardedItemTable(dev(items), id_base=id_base, bf16=mode == MR_SCORE_BF16)
            q = ev.prepare_queries(dev(users), mode=mode)
            for lab in (labels, outside):
                exact = ev.label_ranks(q, table, dev(lab), mode=mode)
                for max_live in (0.0, 1.0):
                    monkeypatch.setattr(evm, "COMPACT_MAX_LIVE", max_live)
                    for cap in (3, 100, N + 1):
                        got = ev.label_ranks(q, table, dev(lab), mode=mode, cap=cap)
                        assert_bounded(got, exact, cap, f"id_base {id_base} mode {mode} cap {cap}")
            assert (ev.label_ranks(q, table, dev(outside), mode=mode, cap=5).cpu() == -1).all()


def planted_inputs(Q, N, E, seed, frac=0.5, noise=0.5):
    """The bench's inputs at another Q: a fraction of the queries planted near their label item."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    items = torch.nn.functional.normalize(torch.randn(N, E, generator=g, device="cuda"), dim=-1)
    users = torch.randn(Q, E, generator=g, device="cuda")
    labels = torch.randint(0, N, (Q,), generator=g, device="cuda")
    planted = torch.rand(Q, generator=g, device="cuda") < frac
    users = torch.where(planted[:, None], items[labels] + noise * users / E ** 0.5, users)
    return torch.nn.functional.normalize(users, dim=-1), items, labels


@pytest.mark.parametrize("ks", [[10, 100], [1, 5, 128]], ids=["10_100", "1_5_128"])
def test_metrics_equal_the_list_path_at_scale(ks):
    """Config 5 at Q = 4,096: `evaluate_embeddings` == `metrics_from_ids(topk_embeddings)` as Python floats, every
    mode, with and without exclusion lists; and with every label its row's top-1 (every row stays live)."""
    Q, N, E = 4096, 1_000_000, 768
    users, items, labels = planted_inputs(Q, N, E, seed=251)
    g = torch.Generator(device="cuda").manual_seed(252)
    ex = torch.randint(-1, N, (Q, 50), generator=g, device="cuda")
    ex[::9, 3] = labels[::9]
    ev = Evaluator(["RECALL", "NDCG"], ks)
    for mode in MODES:
        table = ShardedItemTable(items, bf16=mode == MR_SCORE_BF16)
        for lab, users_ in ((labels, users), (labels, items[labels])):      # the second: every label is the top-1
            q = ev.prepare_queries(users_, mode=mode)
            for exclude in (None, ex):
                want = ev.metrics_from_ids(ev.topk_embeddings(q, table, max(ks), mode=mode, exclude=exclude)[1], lab)
                assert ev.evaluate_embeddings(q, table, lab, mode=mode, exclude=exclude) == want, f"mode {mode}"
        del table


def test_emulated_shards_reproduce_the_one_table_bounded_ranks():
    """World 2, 3 and 8 played by hand: per-shard probes summed, the live rows (sum below the cap) counted against the
    rest of every shard and summed -- the one-table bounded ranks, exact below the cap."""
    Q, N, E, cap = 300, 20011, 64, 50
    users, items, _ = synth.make_catalog(Q, N, E, kind="gauss", seed=261)
    scores = orc.scores_f32(users, items)
    labels = make_labels(scores, 0, seed=262)
    ex = dev(make_histories(scores, 20, labels, 0, seed=263))
    ev = Evaluator(["RECALL"], [10])
    tl = dev(labels)
    for mode in MODES:
        bf16 = mode == MR_SCORE_BF16
        q = ev.prepare_queries(dev(users), mode=mode)
        one = ShardedItemTable(dev(items), bf16=bf16)
        key = label_score(q.hi, q.lo, one, tl, mode)
        for exclude in (None, ex):
            exact = ev.label_ranks(q, one, tl, mode=mode, exclude=exclude)
            want = ev.label_ranks(q, one, tl, mode=mode, exclude=exclude, cap=cap)
            assert_bounded(want, exact, cap)
            csr = None if exclude is None else exclusion_csr(exclude, Q)
            for world in (2, 3, 8):
                tables = [ShardedItemTable(dev(items[a:b]), id_base=a, n_total=N, bf16=bf16)
                          for a, b in (shard_bounds(N, world, r) for r in range(world))]
                n1 = [evm._probe_rows(t.n_local) for t in tables]
                probe = torch.stack([score_rank(q.hi, q.lo, t, tl, key, mode, csr, rows=(0, m))
                                     for t, m in zip(tables, n1)]).sum(dim=0, dtype=torch.int32)
                live = torch.nonzero((key != 0) & (probe < cap)).flatten()
                csr_l = None if exclude is None else exclusion_csr(exclude[live], live.numel())
                lo = None if q.lo is None else q.lo[live].contiguous()
                hi_l, tl_l, key_l = (x[live].contiguous() for x in (q.hi, tl, key))
                rest = torch.stack([score_rank(hi_l, lo, t, tl_l, key_l, mode, csr_l, rows=(m, t.n_local))
                                    for t, m in zip(tables, n1)]).sum(dim=0, dtype=torch.int32)
                got = probe.clone()
                got[live] += rest
                got = torch.where(key == 0, torch.full_like(got, -1), got)
                got = evm._exclusion_miss(got, tl, exclude)
                assert_bounded(got, exact, cap, f"world {world} mode {mode}")
                below = (exact >= 0) & (exact < cap)
                assert torch.equal(got[below], want[below])
