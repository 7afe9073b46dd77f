"""CPU: the label-rank entry points (`mr_label_score`, `mr_score_rank`, `mr_rank_rows`) reject malformed arguments before
any CUDA call, the workspace query is plain arithmetic, and the NDCG gain table is built only as far as the hits reach."""
import numpy as np
import pytest
import torch

from mergerec_b200 import _lib
from mergerec_b200.evaluator import metrics

D = 1 << 20     # a dummy device pointer: never dereferenced, the arguments are rejected first


def label_score(Q=4, N=256, E=32, mode=0):
    return _lib.load().mr_label_score(D, D, Q, D, D, N, E, 0, mode, D, D, D, 1 << 30, None)


def score_rank(Q=4, N=256, E=32, mode=0, off=None, ids=None):
    return _lib.load().mr_score_rank(D, D, Q, D, D, N, E, 0, mode, D, D, off, ids, D, D, 1 << 30, None)


def rank_rows(Q=4, N=256, ld=256, off=None, ids=None):
    return _lib.load().mr_rank_rows(D, Q, N, ld, 0, D, off, ids, D, None)


def rejected(rc, word):
    return rc == -1 and word in _lib.load().mr_last_error()


def test_half_given_exclusion_lists_rejected():
    assert rejected(score_rank(off=D), b"both")
    assert rejected(score_rank(ids=D), b"both")
    assert rejected(rank_rows(off=D), b"both")
    assert rejected(rank_rows(ids=D), b"both")


def test_shape_and_mode_errors():
    for fn in (label_score, score_rank):
        assert rejected(fn(E=30), b"multiple of 4")
        assert rejected(fn(E=36, mode=2), b"multiple of 8")
        assert rejected(fn(Q=-1), b"Q, N >= 0")
        assert rejected(fn(N=-1), b"Q, N >= 0")
        assert rejected(fn(E=0), b"E >= 1")
        assert rejected(fn(mode=7), b"unknown mode")
    assert rejected(rank_rows(Q=-1), b"Q >= 0")
    assert rejected(rank_rows(N=-1), b"N >= 0")
    assert rejected(rank_rows(ld=100), b"ld >= N")


def test_null_pointers_rejected():
    lib = _lib.load()
    assert lib.mr_label_score(D, D, 4, D, D, 256, 32, 0, 0, None, D, D, 1 << 30, None) == -1
    assert lib.mr_label_score(D, None, 4, D, D, 256, 32, 0, 0, D, D, D, 1 << 30, None) == -1   # 3xTF32 needs lo
    assert lib.mr_score_rank(D, D, 4, D, D, 256, 32, 0, 0, D, None, None, None, D, D, 1 << 30, None) == -1
    assert lib.mr_rank_rows(D, 4, 256, 256, 0, None, None, None, D, None) == -1
    # nothing to do: no pointer is needed
    assert lib.mr_score_rank(None, None, 0, None, None, 256, 32, 0, 0, None, None, None, None, None, None, 0, None) == 0
    assert lib.mr_rank_rows(None, 0, 256, 256, 0, None, None, None, None, None) == 0


def test_workspace_query():
    lib = _lib.load()
    assert lib.mr_score_rank_workspace_bytes(0, 1000, 64) == 0
    assert lib.mr_score_rank_workspace_bytes(-1, 1000, 64) < 0
    assert lib.mr_score_rank_workspace_bytes(4, -1, 64) < 0
    assert lib.mr_score_rank_workspace_bytes(4, 1000, 0) < 0
    for Q, N, E in ((1, 1, 4), (300, 20011, 64), (65536, 1_000_000, 768)):
        b = lib.mr_score_rank_workspace_bytes(Q, N, E)
        assert b >= 2 * Q * E * 4 + 256         # the gathered (hi, lo) label rows of the label-score pass
        assert b >= Q * 4                       # at least one count per row
        assert lib.mr_score_rank_workspace_bytes(Q, 0, E) == lib.mr_score_rank_workspace_bytes(Q, 1, E)   # N = 0 plans as 1
    # too small a workspace is a clean argument error, found before any launch
    rc = lib.mr_label_score(D, D, 4, D, D, 256, 32, 0, 0, D, D, D, 16, None)
    assert rc < 0 and b"workspace" in lib.mr_last_error()


def test_gain_table_built_only_to_the_largest_hit():
    t = metrics._gain_table(64)
    for r in (0, 1, 7, 63):
        assert t[r] == 1 / (torch.log2(torch.tensor(r + 2)).item())
    before = metrics._GAINS.size
    ranks = np.array([0, 5, -1, 3000, 20_000, 17], np.int32)
    n = ranks.size
    k = 10 ** 7
    got = metrics.ndcg_from_ranks(ranks, k)
    assert metrics._GAINS.size <= max(before, 20_001)
    want = sum(1 / (torch.log2(torch.tensor(int(r) + 2)).item()) for r in ranks if r >= 0) / n
    assert got == want
    small = np.array([0, 5, -1, 3000, 17], np.int32)
    assert metrics.ndcg_from_found(small[small >= 0], small.size, 10 ** 6) == metrics.ndcg_from_ranks(small, 10 ** 6)
    assert metrics._GAINS.size >= 3001
    # the entries are those of the table built in one go
    assert np.array_equal(metrics._gain_table(1024)[:64], t)
