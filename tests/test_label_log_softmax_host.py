"""CPU: the log-softmax entry points (`mr_score_lse`, `mr_lse_finish`) reject malformed arguments before any CUDA call,
the workspace query is plain arithmetic, and `catalog_cross_entropy` rejects labels outside the catalog."""
import pytest
import torch

from mergerec_b200 import _lib

D = 1 << 20     # a dummy device pointer: never dereferenced, the arguments are rejected first


def score_lse(Q=4, N=256, E=32, mode=0, T=1.0, off=None, ids=None, shift=D, sums=D, ws_bytes=1 << 30):
    return _lib.load().mr_score_lse(D, D, Q, D, D, N, E, 0, mode, T, off, ids, shift, sums, D, ws_bytes, None)


def lse_finish(P=2, Q=4, T=1.0, shift=D, sums=D, key=D, logp=D):
    return _lib.load().mr_lse_finish(shift, sums, P, Q, key, T, logp, None)


def rejected(rc, word):
    return rc == -1 and word in _lib.load().mr_last_error()


def test_half_given_exclusion_lists_rejected():
    assert rejected(score_lse(off=D), b"both")
    assert rejected(score_lse(ids=D), b"both")


def test_temperature_must_be_finite_and_positive():
    for T in (0.0, -1.0, float("inf"), float("nan")):
        assert rejected(score_lse(T=T), b"temperature")
        assert rejected(lse_finish(T=T), b"temperature")


def test_shape_and_mode_errors():
    assert rejected(score_lse(E=30), b"multiple of 4")
    assert rejected(score_lse(E=36, mode=2), b"multiple of 8")
    assert rejected(score_lse(Q=-1), b"Q, N >= 0")
    assert rejected(score_lse(N=-1), b"Q, N >= 0")
    assert rejected(score_lse(E=0), b"E >= 1")
    assert rejected(score_lse(mode=7), b"unknown mode")
    assert rejected(lse_finish(P=-1), b"P < 2^20")
    assert rejected(lse_finish(Q=-1), b"Q >= 0")


def test_null_pointers_rejected():
    lib = _lib.load()
    assert rejected(score_lse(shift=None), b"null pointer")
    assert rejected(score_lse(sums=None), b"null pointer")
    assert lib.mr_score_lse(D, None, 4, D, D, 256, 32, 0, 0, 1.0, None, None, D, D, D, 1 << 30, None) == -1  # 3xTF32: lo
    assert rejected(lse_finish(key=None), b"null pointer")
    assert rejected(lse_finish(logp=None), b"null pointer")
    assert rejected(lse_finish(shift=None), b"null pointer")
    # nothing to do: no pointer is needed
    assert lib.mr_score_lse(None, None, 0, None, None, 256, 32, 0, 0, 1.0, None, None, None, None, None, 0, None) == 0
    assert lse_finish(Q=0, shift=None, sums=None, key=None, logp=None) == 0


def test_workspace_query():
    lib = _lib.load()
    assert lib.mr_score_lse_workspace_bytes(0, 1000, 64) == 0
    assert lib.mr_score_lse_workspace_bytes(-1, 1000, 64) < 0
    assert lib.mr_score_lse_workspace_bytes(4, -1, 64) < 0
    assert lib.mr_score_lse_workspace_bytes(4, 1000, 0) < 0
    for Q, N, E in ((1, 1, 4), (300, 20011, 64), (65536, 1_000_000, 768)):
        b = lib.mr_score_lse_workspace_bytes(Q, N, E)
        assert b >= Q * 12 + 256                 # at least one (shift, sum) pair per row
        assert lib.mr_score_lse_workspace_bytes(Q, 0, E) == lib.mr_score_lse_workspace_bytes(Q, 1, E)   # N = 0 plans as 1
    rc = score_lse(ws_bytes=16)
    assert rc < 0 and b"workspace" in lib.mr_last_error()


def test_catalog_cross_entropy_rejects_labels_outside_the_catalog():
    from mergerec_b200.module.recommender.module import catalog_cross_entropy
    users, items = torch.zeros(3, 8), torch.zeros(10, 8)
    for bad in ([0, 1, 10], [-1, 0, 1]):
        with pytest.raises(ValueError, match="item ids"):
            catalog_cross_entropy(users, items, torch.tensor(bad), 0.05)
