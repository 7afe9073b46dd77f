"""GPU: items left out of each query's ranking (`exclude`, e.g. the user's history) -- the fused scoring kernel
(`mr_score_topk_exclude`), the materialised-matrix path (`mr_topk_rows_exclude`) and every evaluator entry point on top
of them.

Bit-exact bar: on exact-grid catalogs every list must equal the canonical (score desc, id asc) ranking of the eligible
items, padded with (-inf, -1); at scale, exclusion must not change a single score, so the filtered list is a slice of
the unfiltered one."""
import numpy as np
import pytest
import torch

from helpers import assert_bit_equal
from mergerec_b200 import synth
from mergerec_b200.evaluator import Evaluator, ShardedItemTable, shard_bounds
from mergerec_b200.evaluator.evaluator import score_topk, topk_rows
from mergerec_b200.evaluator.sharded import MR_SCORE_BF16, MR_SCORE_TF32X1, MR_SCORE_TF32X3, split_tf32, topk_merge
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

ID_BASE = 1000


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().cpu().numpy()


def oracle_topk(scores, k, exclude, id_base=0):
    """Canonical top-k of each row over the items not in its `exclude` row (negatives = padding), padded with
    (-inf, -1)."""
    Q, N = scores.shape
    vals = np.full((Q, k), -np.inf, np.float32)
    ids = np.full((Q, k), -1, np.int32)
    gid = np.arange(N, dtype=np.int64) + id_base
    for q in range(Q):
        keep = ~np.isin(gid, exclude[q][exclude[q] >= 0])
        s, g = scores[q, keep], gid[keep]
        o = np.lexsort((g, -s))[:k]
        vals[q, :o.size], ids[q, :o.size] = s[o], g[o]
    return vals, ids


def make_histories(scores, k, labels, id_base, seed):
    """One exclusion row per query, cycling through the cases the kernel has to get right (global ids, -1 padding)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    Q, N = scores.shape
    H = min(N, 600) + 12
    ex = np.full((Q, H), -1, np.int64)
    top = oracle_topk(scores, min(k, N), np.full((Q, 1), -1), id_base)[1]
    for q in range(Q):
        case = q % 8 if Q >= 8 else 7 - q
        if case == 0:
            row = []                                                            # nothing excluded
        elif case == 1:                                                         # duplicates, ids of other shards / past N
            r = rng.integers(0, N, 10) + id_base
            row = list(r) + list(r[:4]) + [id_base + N, id_base + N + 7, 2 ** 31 - 1, 0, id_base - 1]
        elif case == 2:                                                         # padding in the middle of the row
            row = list(rng.integers(0, N, 12) + id_base)
            row[3] = row[7] = -1
            row[9] = -5
        elif case == 3:                                                         # the label and some of the best items
            row = [int(labels[q])] + list(top[q, ::2])
        elif case == 4:                                                         # one whole 256-item tile
            t = min(1, (N - 1) // 256)
            row = list(range(id_base + 256 * t, id_base + min(N, 256 * (t + 1))))
        elif case == 5:                                                         # leaves fewer than k items (if N allows)
            row = list(rng.permutation(N)[:max(N - k // 2, 0)] + id_base) if N <= 600 else list(range(id_base, id_base + 600))
        elif case == 6:                                                         # every item (if N allows)
            row = list(range(id_base, id_base + N)) if N <= 600 else list(rng.integers(0, N, 600) + id_base)
        else:                                                                   # the row's own unfiltered top-k
            row = list(rng.permutation(top[q]))
        row = row[:H]
        ex[q, :len(row)] = row
    return ex


def fused(users, items, k, mode, exclude, id_base=ID_BASE):
    table = ShardedItemTable(dev(items), id_base=id_base)
    u_hi, u_lo = split_tf32(dev(users))
    v, i = score_topk(u_hi, u_lo, table, k, mode, exclude=None if exclude is None else dev(exclude))
    return host(v), host(i)


FUSED_SHAPES = [   # the fused-kernel shapes of test_eval_gpu.py: partial query blocks and tiles, E % 32 != 0
    (64, 500, 32, 10), (200, 3000, 64, 100), (257, 1025, 36, 50), (1, 256, 8, 1), (300, 70000, 128, 128),
]


@pytest.mark.parametrize("splits", [0, 3])
@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("shape", FUSED_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_exclude_grid_vs_oracle(shape, cg, splits, monkeypatch):
    """Fused kernel (3xTF32 and 1xTF32, CTA pairs or single CTAs, automatic or 3 item splits -- so lists straddle unit
    boundaries) and the matrix path, against the oracle: ids and score bits."""
    monkeypatch.setenv("MR_SCORE_CTA_GROUP", str(cg))
    monkeypatch.setenv("MR_SCORE_SPLITS", str(splits))
    Q, N, E, k = shape
    users, items, labels = synth.make_catalog(Q, N, E, kind="grid", seed=61)
    scores = orc.scores_f32(users, items)
    ex = make_histories(scores, k, labels + ID_BASE, ID_BASE, seed=62)
    ov, oi = oracle_topk(scores, k, ex, ID_BASE)
    for mode in (MR_SCORE_TF32X3, MR_SCORE_TF32X1):
        v, i = fused(users, items, k, mode, ex)
        assert np.array_equal(i, oi), f"ids, mode {mode}"
        assert_bit_equal(v, ov, f"scores, mode {mode}")
    if splits == 0 and cg == 2:
        v, i = topk_rows(dev(scores), k, id_base=ID_BASE, exclude=dev(ex))
        assert np.array_equal(host(i), oi), "matrix path ids"
        assert_bit_equal(host(v), ov, "matrix path scores")


def big_gauss(Q, N, E, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    users = torch.nn.functional.normalize(torch.randn(Q, E, generator=g, device="cuda"), dim=-1)
    items = torch.nn.functional.normalize(torch.randn(N, E, generator=g, device="cuda"), dim=-1)
    return users, items


@pytest.mark.parametrize("mode", [MR_SCORE_TF32X3, MR_SCORE_BF16])
def test_exclude_unfiltered_topk_at_scale(mode):
    """Q = 4,096 against N = 1,000,000 (E = 768): excluding each row's own top-k leaves positions k .. 2k - 1 of the
    unfiltered top-2k, bit for bit (exclusion never changes how a score is computed).  Then random members of the
    unfiltered top-128 plus random ids outside it: the unfiltered list with those ids removed, cut to k."""
    Q, N, E, k = 4096, 1_000_000, 768, 50
    users, items = big_gauss(Q, N, E, seed=71)
    bf16 = mode == MR_SCORE_BF16
    ev = Evaluator(["RECALL"], [k])
    table = ShardedItemTable(items, bf16=bf16)
    queries = ev.prepare_queries(users, mode=mode)
    v2, i2 = ev.topk_embeddings(queries, table, 2 * k, mode=mode)
    v, i = ev.topk_embeddings(queries, table, k, mode=mode, exclude=i2[:, :k])
    assert torch.equal(i, i2[:, k:]) and torch.equal(v.view(torch.int32), v2[:, k:].view(torch.int32))

    v128, i128 = ev.topk_embeddings(queries, table, 128, mode=mode)
    gen = torch.Generator(device="cuda").manual_seed(72)
    drop = torch.rand((Q, 128), generator=gen, device="cuda") < 0.4
    drop[:, 78:] = False                                                           # the last 50 of the 128 stay
    members = torch.where(drop, i128, torch.full_like(i128, -1))
    outside = torch.randint(0, N, (Q, 40), generator=gen, device="cuda", dtype=torch.int32)
    outside[(outside[:, :, None] == i128[:, None, :]).any(-1)] = -1                 # ids outside the top-128 only
    ex = torch.cat([outside, members, outside[:, :5]], dim=1)                      # unsorted, padded, duplicated
    v, i = ev.topk_embeddings(queries, table, k, mode=mode, exclude=ex)
    ex_h, i128_h, v128_h = host(ex), host(i128), host(v128)
    want_i = np.empty((Q, k), np.int32)
    want_v = np.empty((Q, k), np.float32)
    for q in range(Q):
        keep = ~np.isin(i128_h[q], ex_h[q])
        want_i[q], want_v[q] = i128_h[q][keep][:k], v128_h[q][keep][:k]
    assert np.array_equal(host(i), want_i)
    assert_bit_equal(host(v), want_v, "scores after random exclusion")


def test_exclude_nothing_is_a_no_op():
    """All-padding lists and lists of ids outside the catalog give the bits of the call without `exclude`, on the
    fused path and on the matrix path."""
    users, items, _ = synth.make_catalog(300, 20011, 64, kind="grid", seed=81)
    ev = Evaluator(["RECALL"], [50])
    tu, ti = dev(users), dev(items)
    v0, i0 = ev.topk_embeddings(tu, ti)
    pad = torch.full((300, 7), -1, dtype=torch.int64)
    past = torch.full((300, 3), 20011, dtype=torch.int32).cuda()
    for ex in (pad, pad.cuda(), past):
        v, i = ev.topk_embeddings(tu, ti, exclude=ex)
        assert torch.equal(i, i0) and torch.equal(v.view(torch.int32), v0.view(torch.int32))
    scores = dev(orc.scores_f32(users, items))
    rv0, ri0 = topk_rows(scores, 50)
    for ex in (pad, past):
        rv, ri = topk_rows(scores, 50, exclude=ex)
        assert torch.equal(ri, ri0) and torch.equal(rv.view(torch.int32), rv0.view(torch.int32))


def test_exclude_shards_and_streamed_chunks_equal_one_table():
    """Every rank passes the same global-id lists: shards scored separately and merged equal the one-table call
    (2 and 4 emulated ranks); the host-streamed table (chunks shorter than k included) equals it too."""
    Q, N, E, k = 300, 20011, 64, 50
    users, items, labels = synth.make_catalog(Q, N, E, kind="gauss", seed=91)
    scores = orc.scores_f32(users, items)
    ex = make_histories(scores, k, labels, 0, seed=92)
    v1, i1 = fused(users, items, k, MR_SCORE_TF32X3, ex, id_base=0)
    for world in (2, 4):
        pv, pi = [], []
        for r in range(world):
            a, b = shard_bounds(N, world, r)
            v, i = fused(users, items[a:b], k, MR_SCORE_TF32X3, ex, id_base=a)
            pv.append(dev(v))
            pi.append(dev(i))
        mv, mi = topk_merge(torch.stack(pv), torch.stack(pi), k)
        assert np.array_equal(host(mi), i1) and np.array_equal(host(mv).view(np.uint32), v1.view(np.uint32))

    ev = Evaluator(["NDCG", "RECALL"], [10, k])
    tu = dev(users)
    want_v, want_i = ev.topk_embeddings(tu, dev(items), k, exclude=dev(ex))
    assert np.array_equal(host(want_i), i1)
    v, i = ev.topk_embeddings_streamed(tu, torch.from_numpy(items), k, first_rows=1000, max_chunks=7, exclude=dev(ex))
    assert torch.equal(i, want_i) and torch.equal(v.view(torch.int32), want_v.view(torch.int32))
    # a small catalog whose first chunks hold fewer than k rows
    users, items, labels = synth.make_catalog(70, 90, 32, kind="grid", seed=93)
    ex = make_histories(orc.scores_f32(users, items), 50, labels, 0, seed=94)
    tu = dev(users)
    want_v, want_i = ev.topk_embeddings(tu, dev(items), 50, exclude=torch.from_numpy(ex))
    v, i = ev.topk_embeddings_streamed(tu, torch.from_numpy(items), 50, first_rows=16, max_chunks=7, exclude=torch.from_numpy(ex))
    assert torch.equal(i, want_i) and torch.equal(v.view(torch.int32), want_v.view(torch.int32))
    assert ev.evaluate_embeddings_streamed(tu, torch.from_numpy(items), dev(labels), first_rows=16, exclude=dev(ex)) == \
        ev.evaluate_embeddings(tu, dev(items), dev(labels), exclude=dev(ex))


@pytest.mark.parametrize("cg", [1, 2])
def test_exclude_metrics_vs_oracle(cg, monkeypatch):
    """Recall / NDCG with histories (a label inside its row's history counts as a miss) equal the oracle's metrics on
    the oracle's ids, bit for bit, through `evaluate_embeddings` and through `Evaluator.__call__` on the score matrix."""
    monkeypatch.setenv("MR_SCORE_CTA_GROUP", str(cg))
    Q, N, E = 512, 20000, 96
    users, items, labels = synth.make_catalog(Q, N, E, kind="grid", seed=101)
    scores = orc.scores_f32(users, items)
    ex = make_histories(scores, 20, labels, 0, seed=102)
    ex[::5, -1] = labels[::5]                                              # more labels inside their own history
    metrics, ks = ["RECALL", "NDCG"], [1, 5, 20]
    _, oi = oracle_topk(scores, 20, ex, 0)
    want = orc.evaluate_ids(oi, labels, metrics, ks, "test/")
    ev = Evaluator(metrics, ks)
    _, ids = ev.topk_embeddings(dev(users), dev(items), exclude=dev(ex))
    assert np.array_equal(host(ids), oi)
    got = ev.evaluate_embeddings(dev(users), dev(items), dev(labels), metric_prefix="test/", exclude=dev(ex))
    assert list(got.keys()) == list(want.keys()) and got == want
    assert ev(dev(scores), dev(labels), "test/", exclude=dev(ex)) == want
    assert ev.evaluate(dev(scores), dev(labels), "test/", exclude=torch.from_numpy(ex)) == want
    in_history = (ex == labels[:, None]).any(axis=1)
    assert in_history.sum() > Q // 5 and (orc.label_rank(oi, labels)[in_history] == -1).all()
    assert (orc.label_rank(orc.topk_rows(scores, 20)[1], labels)[in_history] >= 0).any(), "some would be hits without exclude"
