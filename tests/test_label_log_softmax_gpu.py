"""GPU: each query's label log-softmax over the whole catalog inside the fused scoring kernel (`mr_score_lse` +
`mr_lse_finish`, `Evaluator.label_log_softmax`) and the catalog cross-entropy built on it.

Oracle: fp64 log-softmax of the exact scores (grid catalogs and integer embeddings, where every mode computes
them exactly; bf16-rounded for the bf16-compat mode) divided by the temperature, over the row's eligible items, taken
at the label.  Tolerance 1e-5 * max(1, |x|): the fp32 terms and ex2.approx."""
import math

import numpy as np
import pytest
import torch

from mergerec_b200 import _lib, synth
from mergerec_b200.evaluator import Evaluator, ShardedItemTable, shard_bounds
from mergerec_b200.evaluator.evaluator import exclusion_csr, label_score, lse_finish, score_lse
from mergerec_b200.evaluator.sharded import MR_SCORE_BF16, MR_SCORE_TF32X1, MR_SCORE_TF32X3
from mergerec_b200.evaluator.metrics import label_rank
from oracle import oracle as orc
from test_exclude_gpu import big_gauss, make_histories
from test_label_rank_gpu import GRID_SHAPES, bf16_round, dev, host, make_labels, score_keys

pytestmark = pytest.mark.gpu

ID_BASE = 1000
MODES = (MR_SCORE_TF32X3, MR_SCORE_TF32X1, MR_SCORE_BF16)
TOL = 1e-5


def oracle_logp(scores, labels, temperature, exclude=None, id_base=0):
    """log_softmax(scores[q, eligible] / T)[label] in fp64, as x[label] - torch.logsumexp(x) (whose special values the
    kernel follows: torch.log_softmax itself turns a whole row with a +inf into NaN); NaN for a label outside the
    catalog, -inf for a label in its own exclusion row."""
    Q, N = scores.shape
    gid = np.arange(N, dtype=np.int64) + id_base
    out = np.full(Q, np.nan)
    for q in range(Q):
        lab = int(labels[q])
        if not id_base <= lab < id_base + N:
            continue
        ex = exclude[q][exclude[q] >= 0] if exclude is not None else np.zeros(0, np.int64)
        if lab in ex:
            out[q] = -np.inf
            continue
        keep = ~np.isin(gid, ex)
        x = torch.from_numpy(scores[q, keep].astype(np.float64) / temperature)
        out[q] = float(x[int(np.nonzero(gid[keep] == lab)[0][0])] - torch.logsumexp(x, 0))
    return out


def assert_close(got, want, tol=TOL, what=""):
    got = np.asarray(got, np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want)), f"{what}: NaN rows differ"
    inf = np.isinf(want)
    assert np.array_equal(got[inf], want[inf]), f"{what}: infinite rows differ"
    fin = np.isfinite(want)
    assert np.isfinite(got[fin]).all(), f"{what}: non-finite where the oracle is finite"
    err = np.abs(got[fin] - want[fin]) / np.maximum(1.0, np.abs(want[fin]))
    assert err.size == 0 or err.max() <= tol, f"{what}: max scaled error {err.max():.3g}"


def with_full_rows(ex, N, id_base, every=13):
    """`ex` plus rows that leave out every item of the table (every `every`-th row, from row 6)."""
    Q = ex.shape[0]
    full = np.full((Q, N), -1, np.int64)
    full[6::every] = np.arange(N) + id_base
    return np.concatenate([ex, full], axis=1)


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("shape", GRID_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_label_log_softmax_grid_vs_oracle(shape, cg, monkeypatch):
    """All three modes, id_base != 0, with and without exclusion lists (labels inside their own history, rows with
    every item left out), labels outside the catalog."""
    monkeypatch.setenv("MR_SCORE_CTA_GROUP", str(cg))
    Q, N, E = shape
    users, items, _ = synth.make_catalog(Q, N, E, kind="grid", seed=211)
    scores = orc.scores_f32(users, items)
    labels = make_labels(scores, ID_BASE, seed=212)
    ex = with_full_rows(make_histories(scores, 20, labels, ID_BASE, seed=213), N, ID_BASE)
    for mode in MODES:
        if mode == MR_SCORE_BF16 and E % 8:
            continue
        s = bf16_round(scores) if mode == MR_SCORE_BF16 else scores
        table = ShardedItemTable(dev(items), id_base=ID_BASE, bf16=mode == MR_SCORE_BF16)
        queries = Evaluator.prepare_queries(dev(users), mode=mode)
        for T in (1.0, 0.05):
            for exclude in (None, ex):
                want = oracle_logp(s, labels, T, exclude, ID_BASE)
                got = Evaluator.label_log_softmax(queries, table, dev(labels), T, mode=mode,
                                                  exclude=None if exclude is None else dev(exclude))
                assert got.dtype == torch.float32 and got.is_cuda
                assert_close(host(got), want, what=f"mode {mode}, T {T}, exclude {exclude is not None}")


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("N", [15, 300])
def test_label_log_softmax_ids_up_to_int32_max(N, cg, monkeypatch):
    """A table whose ids end at 2^31 - 1: the exclusion cursor of the last chunk, past INT32_MAX."""
    monkeypatch.setenv("MR_SCORE_CTA_GROUP", str(cg))
    Q, E = 70, 64
    id_base = 2 ** 31 - 1 - N
    users, items, _ = synth.make_catalog(Q, N, E, kind="grid", seed=221)
    scores = orc.scores_f32(users, items)
    labels = make_labels(scores, id_base, seed=222)
    ex = make_histories(scores, 10, labels, id_base, seed=223)
    ex[ex >= 2 ** 31] = -1
    ex[::4, -1] = id_base + N - 1
    ex = with_full_rows(ex, N, id_base, every=9)
    for mode in MODES:
        s = bf16_round(scores) if mode == MR_SCORE_BF16 else scores
        table = ShardedItemTable(dev(items), id_base=id_base, bf16=mode == MR_SCORE_BF16)
        queries = Evaluator.prepare_queries(dev(users), mode=mode)
        for exclude in (None, ex):
            want = oracle_logp(s, labels, 0.05, exclude, id_base)
            got = Evaluator.label_log_softmax(queries, table, dev(labels), 0.05, mode=mode,
                                              exclude=None if exclude is None else dev(exclude))
            assert_close(host(got), want, what=f"mode {mode}")


def special_catalog(neg_all):
    """E = 16, N = 100.  Item 3 has a NaN component (a NaN column).  Component 0 is +-1e20 for items 10..29 (or, with
    `neg_all`, -1e20 for every item) and for the users of rows 0..7, so their products overflow to +-inf."""
    rng = np.random.Generator(np.random.PCG64(231))
    Q, N, E = 12, 100, 16
    users = rng.standard_normal((Q, E)).astype(np.float32)
    items = rng.standard_normal((N, E)).astype(np.float32)
    users[:, 0] = 0
    items[:, 0] = 0
    users[0:4, 0], users[4:8, 0] = 1e20, -1e20
    if neg_all:
        items[:, 0] = -1e20
    else:
        items[10:20, 0], items[20:30, 0] = 1e20, -1e20
    items[3, 1] = np.nan
    return users, items


@pytest.mark.parametrize("neg_all", [False, True])
def test_special_values_follow_torch(neg_all):
    """NaN and +-inf scores, with the kernel's own score bits as the oracle's input (topk_embeddings(k = N) returns
    every score): an eligible NaN gives NaN, an eligible +inf gives -inf at finite labels and NaN at +inf labels, a
    row of -inf gives NaN (-inf - -inf), as label score minus torch.logsumexp does."""
    users, items = special_catalog(neg_all)
    Q, N = users.shape[0], items.shape[0]
    labels = np.array([0, 3, 12, 25, 40, 15, 3, 22, 3, 50, 99, 60], np.int64)
    ex = np.full((Q, 40), -1, np.int64)
    ex[1::2, 0] = 3                               # the NaN column left out of every second row
    ex[2::4, 1:21] = np.arange(10, 30)            # the +-inf columns left out
    ev = Evaluator(["RECALL"], [10])
    rows_seen = set()
    for mode in MODES:
        table = ShardedItemTable(dev(items), bf16=mode == MR_SCORE_BF16)
        q = ev.prepare_queries(dev(users), mode=mode)
        v, i = ev.topk_embeddings(q, table, N, mode=mode)
        s = np.zeros((Q, N), np.float32)
        np.put_along_axis(s, host(i).astype(np.int64), host(v), axis=1)
        for exclude in (None, ex):
            want = oracle_logp(s, labels, 0.5, exclude)
            got = ev.label_log_softmax(q, table, dev(labels), 0.5, mode=mode,
                                       exclude=None if exclude is None else dev(exclude))
            assert_close(host(got), want, what=f"mode {mode}")
            for r in range(Q):
                keep = ~np.isin(np.arange(N), exclude[r]) if exclude is not None else np.ones(N, bool)
                e = s[r, keep]
                rows_seen.add("nan" if np.isnan(e).any() else "+inf" if (e == np.inf).any()
                              else "-inf" if (e == -np.inf).all() else "finite")
    assert rows_seen >= ({"nan", "+inf", "finite"} if not neg_all else {"nan", "-inf"})


def int_embeddings(Q, N, m):
    """Rising catalog: items[i] = (i // 4096, (i // 64) % 64, i % 64), users = m_q (4096, 64, 1), so that score = m_q * i
    exactly in every mode (every operand is exact in bf16 and TF32, every partial sum in fp32)."""
    i = np.arange(N)
    items = np.zeros((N, 8), np.float32)
    items[:, 0], items[:, 1], items[:, 2] = i // 4096, (i // 64) % 64, i % 64
    users = np.zeros((Q, 8), np.float32)
    users[:, 0], users[:, 1], users[:, 2] = 4096 * m, 64 * m, m
    return users, items


@pytest.mark.parametrize("mode", MODES)
def test_rising_scores_and_wide_logits(mode):
    """(a) Scores that rise (or fall) with the item id: at T = 0.05 every 16-column chunk holds a new maximum 460+ log2
    units above the last, so the shift moves at every chunk.  (b) Integer embeddings whose dot products span +-9,216,
    logits +-1.8e5 at T = 0.05.  Both against the fp64 oracle, with and without exclusion lists."""
    bf16 = mode == MR_SCORE_BF16
    Q, N = 8, 100_000
    m = np.array([1, 2, 3, -1, -2, 1, 3, -3], np.float32)
    users, items = int_embeddings(Q, N, m)
    scores = m[:, None] * np.arange(N, dtype=np.float32)[None, :]      # exact in fp32: |m i| < 2^24
    if bf16:
        scores = bf16_round(scores)       # the scores the bf16-compat mode ranks (plateaus of equal scores)
    rng = np.random.Generator(np.random.PCG64(241))
    labels = np.array([N - 1, N - 17, 0, 0, 5, rng.integers(N), N // 2, 3], np.int64)
    ex = np.full((Q, 50), -1, np.int64)
    ex[::2] = rng.integers(0, N, (Q // 2, 50))
    ex[1, :20] = N - 1 - np.arange(20)                       # the top of a rising row
    table = ShardedItemTable(dev(items), bf16=bf16)
    q = Evaluator.prepare_queries(dev(users), mode=mode)
    for exclude in (None, ex):
        want = oracle_logp(scores, labels, 0.05, exclude)
        got = Evaluator.label_log_softmax(q, table, dev(labels), 0.05, mode=mode,
                                          exclude=None if exclude is None else dev(exclude))
        assert_close(host(got), want, what="rising")

    Q, N, E = 64, 50_000, 64
    users = rng.integers(-12, 13, (Q, E)).astype(np.float32)
    items = rng.integers(-12, 13, (N, E)).astype(np.float32)
    users[0], users[1] = 12, -12
    items[100], items[N - 5] = 12, -12                       # scores +-9,216 in rows 0 and 1
    items[200:210] = np.sign(users[2:12]) * 12               # near the largest score in rows 2..11
    scores = orc.scores_f32(users, items)
    assert np.abs(scores).max() == 9216
    s = bf16_round(scores) if bf16 else scores
    labels = rng.integers(0, N, Q)
    labels[:12] = [100, N - 5, *range(200, 210)]
    ex = make_histories(scores, 20, labels, 0, seed=242)
    table = ShardedItemTable(dev(items), bf16=bf16)
    q = Evaluator.prepare_queries(dev(users), mode=mode)
    for exclude in (None, ex):
        want = oracle_logp(s, labels, 0.05, exclude)
        got = Evaluator.label_log_softmax(q, table, dev(labels), 0.05, mode=mode,
                                          exclude=None if exclude is None else dev(exclude))
        assert_close(host(got), want, what="wide")


def test_shards_reproduce_the_unsharded_result():
    """Emulated ranks (`shard_bounds` at world sizes 2, 3 and 8): the MAX of the label keys, each shard's partial, and
    `lse_finish` over the stacked partials in rank order equal the one-table result within 1e-6 * max(1, |x|); every
    rank, merging the same gathered partials, holds the same bits."""
    Q, N, E = 300, 20011, 64
    users, items, _ = synth.make_catalog(Q, N, E, kind="gauss", seed=251)
    scores = orc.scores_f32(users, items)
    labels = make_labels(scores, 0, seed=252)
    ex = make_histories(scores, 20, labels, 0, seed=253)
    tl = dev(labels)
    for mode in MODES:
        bf16 = mode == MR_SCORE_BF16
        q = Evaluator.prepare_queries(dev(users), mode=mode)
        for exclude in (None, ex):
            want = host(Evaluator.label_log_softmax(q, ShardedItemTable(dev(items), bf16=bf16), tl, 0.05, mode=mode,
                                                    exclude=None if exclude is None else dev(exclude)))
            csr = None if exclude is None else exclusion_csr(dev(exclude), Q)
            for world in (2, 3, 8):
                tables = [ShardedItemTable(dev(items[a:b]), id_base=a, n_total=N, bf16=bf16)
                          for a, b in (shard_bounds(N, world, r) for r in range(world))]
                keys = [label_score(q.hi, q.lo, t, tl, mode).to(torch.int64) & 0xFFFFFFFF for t in tables]
                key = torch.stack(keys).max(dim=0).values
                key32 = torch.where(key >= 1 << 31, key - (1 << 32), key).to(torch.int32)
                parts = [score_lse(q.hi, q.lo, t, 0.05, mode, csr) for t in tables]
                shift = torch.stack([p[0] for p in parts])
                sums = torch.stack([p[1] for p in parts])
                ranks = [lse_finish(shift, sums, key32, 0.05) for _ in range(world)]
                for r in ranks[1:]:
                    assert torch.equal(r.view(torch.int32), ranks[0].view(torch.int32))
                got = host(ranks[0]).astype(np.float64)
                if exclude is not None:
                    got[(exclude == labels[:, None]).any(1) & (host(key) != 0)] = -np.inf
                assert_close(got, want.astype(np.float64), tol=1e-6, what=f"world {world}, mode {mode}")


def test_lse_partial_of_an_empty_table_and_empty_rows():
    """N = 0 writes the empty partial (shift -2^24, sum 0); a row with every item left out gets the same."""
    Q, E = 5, 32
    users = dev(np.ones((Q, E), np.float32))
    q = Evaluator.prepare_queries(users)
    empty = ShardedItemTable(dev(np.zeros((0, E), np.float32)))
    shift, sums = score_lse(q.hi, q.lo, empty, 1.0)
    assert bool((shift == -(1 << 24)).all()) and bool((sums == 0).all())
    table = ShardedItemTable(dev(np.ones((40, E), np.float32)))
    ex = np.full((Q, 40), -1, np.int64)
    ex[2] = np.arange(40)
    shift, sums = score_lse(q.hi, q.lo, table, 1.0, csr=exclusion_csr(dev(ex), Q))
    assert int(shift[2]) == -(1 << 24) and float(sums[2]) == 0.0
    # every other row: 40 terms of e^32 = 2^(32 log2 e)
    lse = np.delete(host(shift), 2).astype(np.float64) * math.log(2) + np.log(np.delete(host(sums), 2))
    np.testing.assert_allclose(lse, 32 + math.log(40), rtol=1e-6)


def test_at_scale_against_chunked_fp32_scores():
    """Q = 4,096 against N = 1,000,000 (E = 768) Gaussian unit vectors, 3xTF32, T = 0.05, against fp64 log-softmax of
    `mr_scores_fp32` scores (taken in row chunks): within 2 eps / T, eps = 1e-5 the score-error bound.  Where the label
    is in the fused top-100, its key is the key of the list's value, bit for bit."""
    Q, N, E, T = 4096, 1_000_000, 768, 0.05
    users, items = big_gauss(Q, N, E, seed=261)
    ev = Evaluator(["RECALL"], [100])
    table = ShardedItemTable(items)
    q = ev.prepare_queries(users)
    gen = torch.Generator(device="cuda").manual_seed(262)
    v, i = ev.topk_embeddings(q, table, 100)
    labels = torch.randint(0, N, (Q,), generator=gen, device="cuda", dtype=torch.int64)
    pick = torch.randint(0, 100, (Q,), generator=gen, device="cuda")
    labels[::2] = i[::2].gather(1, pick[::2, None])[:, 0].to(torch.int64)
    got = ev.label_log_softmax(q, table, labels, T)
    lib = _lib.load()
    want = torch.empty(Q, dtype=torch.float64, device="cuda")
    rows = 256
    sc = torch.empty((rows, N), dtype=torch.float32, device="cuda")
    for r0 in range(0, Q, rows):
        _lib.check(lib.mr_scores_fp32(_lib.dptr(users[r0:r0 + rows]), rows, _lib.dptr(items), N, E, _lib.dptr(sc), N,
                                      _lib.stream_handle()), "mr_scores_fp32")
        x = sc.to(torch.float64) / T
        want[r0:r0 + rows] = torch.log_softmax(x, dim=1).gather(1, labels[r0:r0 + rows, None])[:, 0]
    err = (got.to(torch.float64) - want).abs()
    assert float(err.max()) <= 2 * 1e-5 / T, float(err.max())
    pos = label_rank(i, labels)
    hit = pos >= 0
    assert int(hit.sum()) >= Q // 2
    key = label_score(q.hi, q.lo, table, labels)
    lv = v.gather(1, pos.clamp(min=0)[:, None].to(torch.int64))[:, 0]
    assert np.array_equal(host(key).view(np.uint32)[host(hit)], score_keys(host(lv))[host(hit)].astype(np.uint32))


def test_rec_evaluation_bf16_metrics_fp32_loss():
    """`RecEvaluation` with bf16-compat metrics on 9,000 queries (three row chunks of the removed loss path): the loss
    is the fp32 catalog cross-entropy (torch on CPU, 1e-5 relative), the metrics are those of the bf16 mode."""
    from mergerec_b200.module.recommender.module import RecEvaluation, catalog_cross_entropy
    Q, N, E = 9000, 5000, 64
    users, items, labels = synth.make_catalog(Q, N, E, kind="gauss", seed=271)
    ev = Evaluator(["NDCG", "RECALL"], [10, 50])
    rec = RecEvaluation(ev, similarity="dot", temperature=0.05, mode=MR_SCORE_BF16)
    rec.set_item_embeddings(dev(items))
    rec.on_epoch_start()
    for a in range(0, Q, 1024):
        rec.step(dev(users[a:a + 1024]), dev(labels[a:a + 1024]))
    got = rec.on_epoch_end("val")
    loss = got.pop("val/epoch_loss")
    scores = torch.from_numpy(orc.scores_f32(users, items))
    ref = float(torch.nn.functional.cross_entropy(scores / 0.05, torch.from_numpy(labels)))
    assert abs(loss - ref) <= 1e-5 * max(1.0, abs(ref))
    assert got == ev.evaluate_embeddings(dev(users), dev(items), dev(labels), "val/", mode=MR_SCORE_BF16)
    # the loss of the fp32 metric path is the same value: the loss ignores the metrics' mode
    rec32 = RecEvaluation(ev, similarity="dot", temperature=0.05)
    rec32.set_item_embeddings(dev(items))
    rec32.on_epoch_start()
    rec32.step(dev(users), dev(labels))
    assert rec32.on_epoch_end("val")["val/epoch_loss"] == loss
    out = catalog_cross_entropy(dev(users), dev(items), dev(labels), 0.05)
    assert out.dtype == torch.float32 and out.dim() == 0 and out.is_cuda and float(out) == loss
