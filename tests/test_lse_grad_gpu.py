"""GPU: the gradient of `Evaluator.label_log_softmax` with respect to the query embeddings (`mr_score_lse_grad`: the
kEpiProb / kEpiAccum passes of the fused scoring kernel) against fp64 autograd, per row within
max |dU - dU64| <= 5e-5 * max |dU64| of that row; rows without a gradient exactly 0.

The bound is twice the largest error measured over these tests (2.3e-5, NVIDIA B200): the logits carry the forward's
3xTF32 score error divided by T, and W . items is accumulated in fp32 by the tensor core over 2,048-item chunks.  torch's
own fp32-logits autograd is 1.7e-5 from fp64 on the config-5 data of tools/lse_grad_bench.py, where this path is 1.3e-5."""
import warnings

import pytest
import torch

from mergerec_b200.evaluator import MR_SCORE_BF16, MR_SCORE_TF32X1, MR_SCORE_TF32X3, Evaluator, ShardedItemTable
from mergerec_b200.evaluator.evaluator import _ordered_sum, lse_finish, score_lse, score_lse_grad

pytestmark = pytest.mark.gpu
TOL = 5e-5
WORST = {}   # largest observed error / bound per test, printed with -s


def case(Q, N, E, T, seed):
    """Queries scaled so that the logits (score / T) have a spread of about 2: neither uniform nor one-hot."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    items = torch.randn(N, E, device="cuda", generator=gen)
    users = torch.randn(Q, E, device="cuda", generator=gen) * (2.0 * T / E ** 0.5)
    labels = torch.randint(0, N, (Q,), device="cuda", generator=gen)
    g = torch.randn(Q, device="cuda", generator=gen)
    g[::5] = 0.0
    return users, items, labels, g


def make_exclude(Q, N, labels, seed):
    """Random ids with duplicates and padding, row 1's label excluded, and (small catalogs) row 2 excluding everything."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    H = N if N <= 5000 else 64
    ex = torch.randint(0, N, (Q, H), device="cuda", generator=gen)
    if H >= 3:
        ex[:, 1] = ex[:, 0]              # duplicates
        ex[:, -1] = -1                   # padding
    if Q > 1 and H >= 3:
        ex[1, 2] = labels[1]
    if Q > 2 and H == N:
        ex[2] = torch.arange(N, device="cuda")
    return ex


def ref_grad(users, items, labels, T, g, exclude=None, normalize=False):
    """fp64 autograd of sum_q g_q * log_softmax(U64 @ I64.T / T, masked by exclude)[q, labels[q]] over the rows whose
    label is eligible; the other rows have no gradient."""
    Q, N = users.shape[0], items.shape[0]
    mask = torch.zeros(Q, N, dtype=torch.bool, device=users.device)
    if exclude is not None:
        ex = exclude.to(torch.int64)
        rows = torch.arange(Q, device=users.device)[:, None].expand_as(ex)
        keep = ex >= 0
        mask[rows[keep], ex[keep]] = True
    valid = ~mask[torch.arange(Q, device=users.device), labels]
    u = users.double().detach().requires_grad_(True)
    x = torch.nn.functional.normalize(u, p=2, dim=-1) if normalize else u
    s = (x[valid] @ items.double().T) / T
    s = s.masked_fill(mask[valid], -float("inf"))
    logp = torch.log_softmax(s, dim=1).gather(1, labels[valid][:, None])[:, 0]
    (logp * g[valid].double()).sum().backward()
    return u.grad if u.grad is not None else torch.zeros_like(u)


def check_rows(got, want, name):
    """max |got - want| per row <= TOL * max |want| of the row (a row of zeros must be exactly zero)."""
    err = (got.double() - want).abs().max(dim=1).values
    bound = TOL * want.abs().max(dim=1).values
    assert torch.isfinite(got).all(), name
    assert bool((err <= bound).all()), (name, float((err - bound).max()))
    assert bool((err[bound == 0] == 0).all()), name
    nz = bound > 0
    if nz.any():
        WORST[name] = max(WORST.get(name, 0.0), float((err[nz] / bound[nz]).max()) * TOL)
    print(f"{name}: max row error / row max = {WORST.get(name, 0.0):.3g}")


def grad_of(users, items, labels, T, g, exclude=None, normalize=False, item_table=None):
    u = users.clone().requires_grad_(True)
    logp = Evaluator.label_log_softmax(u, items if item_table is None else item_table, labels, T, normalize=normalize,
                                       exclude=exclude)
    logp.backward(g)
    return u.grad, logp


SHAPES = [(1, 1, 4), (37, 1000, 64), (300, 5000, 768), (257, 70001, 1024)]


@pytest.mark.parametrize("Q,N,E", SHAPES)
@pytest.mark.parametrize("T", [0.05, 1.0])
@pytest.mark.parametrize("excl", [False, True])
def test_grad_matches_fp64_autograd(Q, N, E, T, excl):
    users, items, labels, g = case(Q, N, E, T, seed=Q + N + E)
    exclude = make_exclude(Q, N, labels, seed=N) if excl else None
    got, logp = grad_of(users, items, labels, T, g, exclude)
    want = ref_grad(users, items, labels, T, g, exclude)
    check_rows(got, want, f"grad {Q}x{N}x{E} T={T} excl={excl}")
    if excl:
        if Q > 1:
            assert logp[1] == -float("inf") and bool((got[1] == 0).all())    # label excluded: no gradient
        if Q > 2 and N <= 5000:
            assert bool((got[2] == 0).all())                                 # every item excluded


def test_grad_with_normalize_matches_fp64_autograd():
    Q, N, E, T = 200, 3000, 128, 0.05
    users, items, labels, g = case(Q, N, E, T, seed=5)
    users = users * 37.0   # the normalisation has something to undo
    items = torch.nn.functional.normalize(items, dim=-1)
    got, _ = grad_of(users, items, labels, T, g, normalize=True)
    want = ref_grad(users, items, labels, T, g, normalize=True)
    check_rows(got, want, "normalize")


def test_forward_bits_and_repeatable_backward():
    Q, N, E, T = 300, 20011, 256, 0.05
    users, items, labels, g = case(Q, N, E, T, seed=7)
    exclude = make_exclude(Q, N, labels, seed=8)
    plain = Evaluator.label_log_softmax(users, items, labels, T, exclude=exclude)
    a, logp = grad_of(users, items, labels, T, g, exclude)
    b, _ = grad_of(users, items, labels, T, g, exclude)
    assert torch.equal(logp.detach().view(torch.int32), plain.view(torch.int32))
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    # the cross-entropy inherits the gradient through its mean
    from mergerec_b200.module.recommender.module import catalog_cross_entropy
    u = users.clone().requires_grad_(True)
    catalog_cross_entropy(u, items, labels, T).backward()
    want = ref_grad(users, items, labels, T, torch.full((Q,), -1.0 / Q, device="cuda"))
    check_rows(u.grad, want, "cross-entropy")


def test_items_and_prepared_queries_stay_constant():
    Q, N, E, T = 64, 2000, 64, 1.0
    users, items, labels, g = case(Q, N, E, T, seed=9)
    it = items.clone().requires_grad_(True)
    u = users.clone().requires_grad_(True)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        logp = Evaluator.label_log_softmax(u, it, labels, T)
    logp.backward(g)
    assert it.grad is None and u.grad is not None
    import mergerec_b200.evaluator.evaluator as ev
    assert ev._warned_item_grad and (len(w) <= 1)
    q = Evaluator.prepare_queries(users)
    assert not Evaluator.label_log_softmax(q, items, labels, T).requires_grad


@pytest.mark.parametrize("mode", [MR_SCORE_BF16, MR_SCORE_TF32X1])
def test_backward_outside_3xtf32_raises(mode):
    Q, N, E, T = 32, 1000, 64, 1.0
    users, items, labels, g = case(Q, N, E, T, seed=11)
    plain = Evaluator.label_log_softmax(users, items, labels, T, mode=mode)
    u = users.clone().requires_grad_(True)
    logp = Evaluator.label_log_softmax(u, items, labels, T, mode=mode)
    assert torch.equal(logp.detach().view(torch.int32), plain.view(torch.int32))
    with pytest.raises(RuntimeError, match="MR_SCORE_TF32X3"):
        logp.backward(g)


def test_sharded_partials_emulated():
    """Per-shard parts from the merged partials of all shards, summed in rank order: the bits of the sharded
    backward's sum (`_ordered_sum`), within the tolerance of the single table."""
    Q, N, E, T = 129, 30011, 256, 0.05
    users, items, labels, g = case(Q, N, E, T, seed=13)
    exclude = make_exclude(Q, N, labels, seed=14)
    q = Evaluator.prepare_queries(users)
    from mergerec_b200.evaluator.evaluator import _device_csr
    from mergerec_b200.evaluator.sharded import shard_bounds
    csr = _device_csr(exclude, Q, users.device)
    G = 3
    tables = []
    for r in range(G):
        lo, hi = shard_bounds(N, G, r)
        tables.append(ShardedItemTable(items[lo:hi], id_base=lo, n_total=N))
    parts = [score_lse(q.hi, q.lo, t, T, MR_SCORE_TF32X3, csr) for t in tables]
    shift = torch.stack([p[0] for p in parts]).contiguous()
    sums = torch.stack([p[1] for p in parts]).contiguous()
    single = ShardedItemTable(items)
    key = Evaluator._label_key(q, single, labels, MR_SCORE_TF32X3)
    logp = lse_finish(shift, sums, key, T)
    gg = torch.where(logp.isfinite() & (exclude != labels[:, None]).all(dim=1), g, torch.zeros_like(g))
    local = torch.stack([score_lse_grad(q.hi, q.lo, t, T, labels, shift, sums, gg, csr) for t in tables])
    got = _ordered_sum(local)
    manual = local[0] + local[1] + local[2]
    assert torch.equal(got.view(torch.int32), manual.view(torch.int32))
    again = torch.stack([score_lse_grad(q.hi, q.lo, t, T, labels, shift, sums, gg, csr) for t in tables])
    assert torch.equal(again.view(torch.int32), local.view(torch.int32))
    want = ref_grad(users, items, labels, T, g, exclude)
    check_rows(got, want, "sharded x3")


def test_grad_at_scale_against_chunked_fp64():
    """Q = 2048, N = 10^6, E = 768 against a chunked fp64 GPU reference of the same formula."""
    Q, N, E, T = 2048, 1_000_000, 768, 0.05
    users, items, labels, g = case(Q, N, E, T, seed=17)
    got, _ = grad_of(users, items, labels, T, g)
    del _
    U, step = users.double(), 65536
    lse = torch.full((Q,), -float("inf"), dtype=torch.float64, device="cuda")
    for n0 in range(0, N, step):
        lse = torch.logaddexp(lse, torch.logsumexp(U @ items[n0:n0 + step].double().T / T, dim=1))
    acc = torch.zeros(Q, E, dtype=torch.float64, device="cuda")
    for n0 in range(0, N, step):
        I = items[n0:n0 + step].double()
        acc += torch.exp(U @ I.T / T - lse[:, None]) @ I
    want = -(g.double() / T)[:, None] * (acc - items[labels].double())
    check_rows(got, want, "scale 2048x1e6x768")
