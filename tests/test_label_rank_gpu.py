"""GPU: each query's label ranked against the whole catalog -- the two passes inside the fused scoring kernel
(`mr_label_score`, `mr_score_rank`), the materialised-matrix path (`mr_rank_rows`) and the evaluator entry points on top
of them (`Evaluator.label_ranks`, `rank_rows`, `metrics_from_ranks`, large ks).

Exact bar: on grid catalogs every rank must equal the label's position in a lexsort by (score key desc, id asc) over the
eligible items; at scale, wherever the label is in the fused top-128 list, its rank is its position there, and the
label's key is the key of the list's score, bit for bit."""
import numpy as np
import pytest
import torch

from mergerec_b200 import synth
from mergerec_b200.evaluator import Evaluator, ShardedItemTable, shard_bounds
from mergerec_b200.evaluator.evaluator import exclusion_csr, label_score, rank_rows, score_rank
from mergerec_b200.evaluator.metrics import label_rank
from mergerec_b200.evaluator.sharded import MR_SCORE_BF16, MR_SCORE_TF32X1, MR_SCORE_TF32X3
from oracle import oracle as orc
from test_exclude_gpu import big_gauss, make_histories

pytestmark = pytest.mark.gpu

ID_BASE = 1000
MODES = (MR_SCORE_TF32X3, MR_SCORE_TF32X1, MR_SCORE_BF16)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().cpu().numpy()


def bf16_round(s):
    """The bf16-compat mode's rounding of an fp32 score (RN-even), with the kernel's bit operations."""
    b = np.ascontiguousarray(s, np.float32).view(np.uint32).astype(np.uint64)
    fin = (b & 0x7F800000) != 0x7F800000
    b = np.where(fin, b + 0x7FFF + ((b >> 16) & 1), b) & 0xFFFF0000
    return b.astype(np.uint32).view(np.float32)


def score_keys(s):
    """The order-preserving uint32 key of topk_common.cuh: -0 == +0, NaN above everything."""
    u = (np.asarray(s, np.float32) + np.float32(0)).view(np.uint32).astype(np.uint64)
    k = np.where(u & 0x80000000, ~u & 0xFFFFFFFF, u | 0x80000000)
    return np.where(np.isnan(s), 0xFFFFFFFF, k).astype(np.uint64)


def oracle_ranks(scores, labels, exclude=None, id_base=0):
    """Position of each label in a lexsort by (key desc, id asc) over the row's items minus `exclude`; -1 when the label
    is not an item or is excluded."""
    Q, N = scores.shape
    gid = np.arange(N, dtype=np.int64) + id_base
    out = np.full(Q, -1, np.int64)
    for q in range(Q):
        lab = int(labels[q])
        ex = exclude[q][exclude[q] >= 0] if exclude is not None else np.zeros(0, np.int64)
        if not id_base <= lab < id_base + N or lab in ex:
            continue
        keep = ~np.isin(gid, ex)
        k, g = score_keys(scores[q, keep]), gid[keep]
        order = np.lexsort((g, -k.astype(np.float64)))
        out[q] = int(np.nonzero(g[order] == lab)[0][0])
    return out


def make_labels(scores, id_base, seed):
    """Labels in the catalog, tied with many items, negative, below id_base and at / above id_base + N."""
    rng = np.random.Generator(np.random.PCG64(seed))
    Q, N = scores.shape
    lab = rng.integers(0, N, Q) + id_base
    for q in range(Q):
        case = q % 7
        if case == 1:                                          # an item of the row's most common score
            vals, counts = np.unique(scores[q], return_counts=True)
            lab[q] = id_base + int(rng.choice(np.nonzero(scores[q] == vals[np.argmax(counts)])[0]))
        elif case == 2:
            lab[q] = -1 - q
        elif case == 3:
            lab[q] = id_base - 1
        elif case == 4:
            lab[q] = id_base + N + (q % 3)
        elif case == 5:
            lab[q] = id_base + N - 1                           # the last item (partial tile)
    return lab


GRID_SHAPES = [(64, 500, 8), (257, 1025, 36), (300, 200, 768), (130, 3000, 1024), (1, 256, 8)]


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("shape", GRID_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_label_ranks_grid_vs_oracle(shape, cg, monkeypatch):
    """All three modes, with and without exclusion lists, through `label_ranks` and `rank_rows` (the latter on the
    mode's scores: bf16-rounded for bf16-compat); the label keys against the oracle's scores."""
    monkeypatch.setenv("MR_SCORE_CTA_GROUP", str(cg))
    Q, N, E = shape
    users, items, _ = synth.make_catalog(Q, N, E, kind="grid", seed=111)
    scores = orc.scores_f32(users, items)
    labels = make_labels(scores, ID_BASE, seed=112)
    ex = make_histories(scores, 20, labels, ID_BASE, seed=113)
    ev = Evaluator(["RECALL"], [10])
    for mode in MODES:
        if mode == MR_SCORE_BF16 and E % 8:
            continue
        s = bf16_round(scores) if mode == MR_SCORE_BF16 else scores
        table = ShardedItemTable(dev(items), id_base=ID_BASE, bf16=mode == MR_SCORE_BF16)
        queries = ev.prepare_queries(dev(users), mode=mode)
        key = host(label_score(queries.hi, queries.lo, table, dev(labels), mode)).view(np.uint32)
        inside = (labels >= ID_BASE) & (labels < ID_BASE + N)
        want_key = np.zeros(Q, np.uint64)
        want_key[inside] = score_keys(s[np.nonzero(inside)[0], labels[inside] - ID_BASE])
        assert np.array_equal(key.astype(np.uint64), want_key), f"label keys, mode {mode}"
        for exclude in (None, ex):
            want = oracle_ranks(s, labels, exclude, ID_BASE)
            got = ev.label_ranks(queries, table, dev(labels), mode=mode,
                                 exclude=None if exclude is None else dev(exclude))
            assert got.dtype == torch.int32 and np.array_equal(host(got), want), f"fused, mode {mode}"
            if cg == 2:
                got = rank_rows(dev(s), dev(labels), id_base=ID_BASE, exclude=None if exclude is None else dev(exclude))
                assert np.array_equal(host(got), want), f"rank_rows, mode {mode}"


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("N", [15, 300])
def test_label_ranks_ids_up_to_int32_max(N, cg, monkeypatch):
    """A table whose ids end at 2^31 - 1 (id_base + N at the 31-bit limit the entry points accept): its last 16-column
    chunk spans ids past INT32_MAX, and the exclusion cursor must still stop there.  With and without exclusion lists,
    all three modes, against the oracle and `rank_rows`."""
    monkeypatch.setenv("MR_SCORE_CTA_GROUP", str(cg))
    Q, E = 70, 64
    id_base = 2 ** 31 - 1 - N
    users, items, _ = synth.make_catalog(Q, N, E, kind="grid", seed=161)
    scores = orc.scores_f32(users, items)
    labels = make_labels(scores, id_base, seed=162)
    ex = make_histories(scores, 10, labels, id_base, seed=163)
    ex[ex >= 2 ** 31] = -1                                     # ids must fit int32
    ex[::4, -1] = id_base + N - 1                              # the last item of the table
    ev = Evaluator(["RECALL"], [10])
    for mode in MODES:
        s = bf16_round(scores) if mode == MR_SCORE_BF16 else scores
        table = ShardedItemTable(dev(items), id_base=id_base, bf16=mode == MR_SCORE_BF16)
        queries = ev.prepare_queries(dev(users), mode=mode)
        for exclude in (None, ex):
            want = oracle_ranks(s, labels, exclude, id_base)
            xt = None if exclude is None else dev(exclude)
            assert np.array_equal(host(ev.label_ranks(queries, table, dev(labels), mode=mode, exclude=xt)), want)
            assert np.array_equal(host(rank_rows(dev(s), dev(labels), id_base=id_base, exclude=xt)), want)


def test_rank_rows_special_values_strided_and_host():
    """NaN, +-0 and -inf scores (NaN ranks above everything, -0 == +0), a strided view and host inputs."""
    rng = np.random.Generator(np.random.PCG64(121))
    Q, N = 97, 3001
    s = (rng.integers(-4, 5, (Q, N)) / 4).astype(np.float32)
    s[rng.random((Q, N)) < 0.05] = np.nan
    s[rng.random((Q, N)) < 0.05] = -0.0
    s[rng.random((Q, N)) < 0.05] = -np.inf
    s[rng.random((Q, N)) < 0.02] = np.float32(np.inf)
    labels = make_labels(np.nan_to_num(s), 7, seed=122)
    labels[::9] = 7 + np.argmax(np.isnan(s[::9]), axis=1)           # NaN labels
    labels[1::9] = 7 + np.argmax(s[1::9] == 0, axis=1)               # labels scored +-0
    ex = make_histories(np.nan_to_num(s), 20, labels, 7, seed=123)
    for exclude in (None, ex):
        want = oracle_ranks(s, labels, exclude, 7)
        xt = None if exclude is None else torch.from_numpy(exclude)
        assert np.array_equal(host(rank_rows(dev(s), dev(labels), 7, xt)), want)
        assert np.array_equal(host(rank_rows(torch.from_numpy(s), torch.from_numpy(labels), 7, xt)), want)
        wide = np.full((Q, N + 13), 5.0, np.float32)
        wide[:, 3:N + 3] = s
        assert np.array_equal(host(rank_rows(dev(wide)[:, 3:N + 3], dev(labels), 7, xt)), want)


def test_shards_reproduce_the_unsharded_ranks():
    """Emulated ranks (`shard_bounds` at world sizes 2, 3 and 8): each scores the labels it owns, the MAX of the keys
    and the SUM of the counts, played by hand, give the ranks of the one-table call."""
    Q, N, E = 300, 20011, 64
    users, items, _ = synth.make_catalog(Q, N, E, kind="gauss", seed=131)
    scores = orc.scores_f32(users, items)
    labels = make_labels(scores, 0, seed=132)
    ex = make_histories(scores, 20, labels, 0, seed=133)
    ev = Evaluator(["RECALL"], [10])
    tl = dev(labels)
    for mode in MODES:
        bf16 = mode == MR_SCORE_BF16
        q = ev.prepare_queries(dev(users), mode=mode)
        for exclude in (None, ex):
            want = ev.label_ranks(q, ShardedItemTable(dev(items), bf16=bf16), tl, mode=mode,
                                  exclude=None if exclude is None else dev(exclude))
            csr = None if exclude is None else exclusion_csr(dev(exclude), Q)
            for world in (2, 3, 8):
                tables = [ShardedItemTable(dev(items[a:b]), id_base=a, n_total=N, bf16=bf16)
                          for a, b in (shard_bounds(N, world, r) for r in range(world))]
                keys = [label_score(q.hi, q.lo, t, tl, mode).to(torch.int64) & 0xFFFFFFFF for t in tables]
                key = torch.stack(keys).max(dim=0).values
                assert int((torch.stack(keys) != 0).sum()) == int((key != 0).sum())    # one owner per label
                key32 = torch.where(key >= 1 << 31, key - (1 << 32), key).to(torch.int32)     # the uint32 bits
                counts = torch.stack([score_rank(q.hi, q.lo, t, tl, key32, mode, csr) for t in tables]).sum(dim=0)
                got = torch.where(key == 0, torch.full_like(counts, -1), counts)
                if exclude is not None:
                    got[torch.from_numpy((exclude == labels[:, None]).any(1)).cuda()] = -1
                assert torch.equal(got.to(torch.int32), want), f"world {world}, mode {mode}"


@pytest.mark.parametrize("mode", MODES)
def test_ranks_agree_with_the_fused_lists_at_scale(mode):
    """Q = 4,096 against N = 1,000,000 (E = 768): where the label is in the K = 128 fused list, its rank is its
    position there and its key is the key of the list's score; elsewhere the rank is >= 128 or -1.  Metrics from
    the ranks equal `evaluate_embeddings`' as floats.  With and without a 50-id exclusion per query."""
    Q, N, E = 4096, 1_000_000, 768
    users, items = big_gauss(Q, N, E, seed=141)
    bf16 = mode == MR_SCORE_BF16
    ks = [1, 10, 50, 100, 128]
    ev = Evaluator(["RECALL", "NDCG"], ks)
    table = ShardedItemTable(items, bf16=bf16)
    q = ev.prepare_queries(users, mode=mode)
    gen = torch.Generator(device="cuda").manual_seed(142)
    v0, i0 = ev.topk_embeddings(q, table, 128, mode=mode)
    pick = torch.randint(0, 128, (Q,), generator=gen, device="cuda")
    labels = torch.randint(0, N, (Q,), generator=gen, device="cuda", dtype=torch.int64)
    labels[::2] = i0[::2].gather(1, pick[::2, None])[:, 0].to(torch.int64)      # half the labels inside the list
    labels[3::16] = i0[3::16, 0].to(torch.int64)                                 # and some at position 0
    excl = torch.randint(0, N, (Q, 50), generator=gen, device="cuda", dtype=torch.int64)
    excl[:, :10] = i0[:, 5:15]                                                   # some of the best items
    excl[7::11, 20] = labels[7::11]                                              # labels inside their own history
    for exclude in (None, excl):
        v, i = ev.topk_embeddings(q, table, 128, mode=mode, exclude=exclude)
        ranks = ev.label_ranks(q, table, labels, mode=mode, exclude=exclude)
        pos = label_rank(i, labels)
        hit = pos >= 0
        assert torch.equal(ranks[hit], pos[hit])
        assert bool(((ranks[~hit] >= 128) | (ranks[~hit] == -1)).all())
        assert int(hit.sum()) > Q // 4
        key = label_score(q.hi, q.lo, table, labels, mode)
        lv = v.gather(1, pos.clamp(min=0)[:, None].to(torch.int64))[:, 0]
        want_key = score_keys(host(lv))
        assert np.array_equal(host(key).view(np.uint32)[host(hit)], want_key[host(hit)].astype(np.uint32))
        assert ev.metrics_from_ranks(ranks) == ev.evaluate_embeddings(q, table, labels, mode=mode, exclude=exclude)
        if exclude is not None:
            assert bool((ranks[7::11] == -1).all())


def test_large_k_metrics_vs_oracle():
    """`evaluate_embeddings` with ks = [10, 200, 1000, N] and `__call__` with ks up to N equal the oracle's floats
    (oracle: the reference metrics on the full canonical ranking)."""
    Q, N, E = 300, 5000, 64
    users, items, labels = synth.make_catalog(Q, N, E, kind="grid", seed=151)
    scores = orc.scores_f32(users, items)
    ex = make_histories(scores, 20, labels, 0, seed=152)
    metrics = ["RECALL", "NDCG"]
    _, full_ids = orc.topk_rows(scores, N)
    for exclude in (None, ex):
        ids = full_ids
        if exclude is not None:
            ids = np.array([np.concatenate([r[~np.isin(r, e[e >= 0])], np.full(np.isin(r, e[e >= 0]).sum(), -1)])
                            for r, e in zip(full_ids, exclude)])
        xt = None if exclude is None else dev(exclude)
        for ks in ([10, 200, 1000, N], [5, 1024, 1025, 4000, N]):
            want = orc.evaluate_ids(ids, labels, metrics, ks, "test/")
            ev = Evaluator(metrics, ks)
            assert ev.evaluate_embeddings(dev(users), dev(items), dev(labels), "test/", exclude=xt) == want
            assert ev(dev(scores), dev(labels), "test/", exclude=xt) == want
            assert ev.evaluate(torch.from_numpy(scores), torch.from_numpy(labels), "test/", exclude=xt) == want
    with pytest.raises(RuntimeError):
        Evaluator(metrics, [N + 1]).evaluate_embeddings(dev(users), dev(items), dev(labels))
    with pytest.raises(RuntimeError):
        Evaluator(metrics, [N + 1])(dev(scores), dev(labels))
