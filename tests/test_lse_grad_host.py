"""CPU: the log-softmax gradient entry point (`mr_score_lse_grad`) rejects malformed arguments before any CUDA call, and
its workspace query is plain arithmetic."""
from mergerec_b200 import _lib

D = 1 << 20     # a dummy device pointer: never dereferenced, the arguments are rejected first


def lse_grad(Q=4, N=256, E=32, T=1.0, off=None, ids=None, labels=D, shift=D, sums=D, P=1, g=D, dU=D, lo=D,
             ws_bytes=1 << 40):
    return _lib.load().mr_score_lse_grad(D, lo, Q, D, lo, N, E, 0, T, off, ids, labels, shift, sums, P, g, dU, D, ws_bytes,
                                         None)


def rejected(rc, word):
    return rc == -1 and word in _lib.load().mr_last_error()


def test_half_given_exclusion_lists_rejected():
    assert rejected(lse_grad(off=D), b"both")
    assert rejected(lse_grad(ids=D), b"both")


def test_temperature_and_partials():
    for T in (0.0, -1.0, float("inf"), float("nan")):
        assert rejected(lse_grad(T=T), b"temperature")
    assert rejected(lse_grad(P=0), b"P < 2^20")
    assert rejected(lse_grad(P=1 << 20), b"P < 2^20")


def test_shape_errors():
    assert rejected(lse_grad(E=30), b"multiple of 4")
    assert rejected(lse_grad(Q=-1), b"Q, N >= 0")
    assert rejected(lse_grad(N=-1), b"Q, N >= 0")
    assert rejected(lse_grad(E=0), b"E >= 1")


def test_null_pointers_rejected():
    for name in ("labels", "shift", "sums", "g", "dU"):
        assert rejected(lse_grad(**{name: None}), b"null pointer"), name
    assert rejected(lse_grad(lo=None), b"lo operands")   # 3xTF32 only: the lo operands are required
    lib = _lib.load()
    # nothing to add: no pointer is needed
    assert lib.mr_score_lse_grad(None, None, 0, None, None, 256, 32, 0, 1.0, None, None, None, None, None, 1, None, None,
                                 None, 0, None) == 0


def test_misaligned_gradient_rejected():
    assert rejected(lse_grad(dU=D + 4), b"aligned")


def test_workspace_query():
    lib = _lib.load()
    assert lib.mr_score_lse_grad_workspace_bytes(0, 1000, 64) == 0
    assert lib.mr_score_lse_grad_workspace_bytes(4, 0, 64) == 0
    assert lib.mr_score_lse_grad_workspace_bytes(-1, 1000, 64) < 0
    assert lib.mr_score_lse_grad_workspace_bytes(4, -1, 64) < 0
    assert lib.mr_score_lse_grad_workspace_bytes(4, 1000, 0) < 0
    for Q, N, E in ((1, 1, 4), (300, 20011, 64), (4096, 1_000_000, 768), (65536, 1_000_000, 768)):
        b = lib.mr_score_lse_grad_workspace_bytes(Q, N, E)
        # the merged normaliser, and W plus the transposed chunk (hi, lo) of at least one 256-item tile
        assert b >= Q * 12 + (Q + E) * 256 * 8
        # bounded by the chunk, not by the catalog: never the (Q, N) matrix
        assert b < Q * 12 + (Q + E) * 65536 * 8 + (1 << 24)
        assert b <= lib.mr_score_lse_grad_workspace_bytes(Q, 2 * N, E)
    rc = lse_grad(ws_bytes=16)
    assert rc < 0 and b"workspace" in lib.mr_last_error()
