"""CPU: the exclusion lists of the evaluator -- the (Q, H) padded-id tensor -> CSR conversion, and the argument checks
of the two exclusion entry points, which reject NULL lists before any CUDA call."""
import numpy as np
import pytest
import torch

from mergerec_b200 import _lib
from mergerec_b200.evaluator.evaluator import exclusion_csr


def rows_of(off, ids):
    off, ids = off.tolist(), ids.tolist()
    return [ids[off[q]:off[q + 1]] for q in range(len(off) - 1)]


def test_csr_padding_duplicates_order_and_empty_rows():
    ex = torch.tensor([[7, -1, 3, 3, 12],
                       [-1, -1, -1, -1, -1],
                       [5, 4, -3, 2, -1],
                       [0, 2 ** 31 - 1, 1, -1, 0]], dtype=torch.int64)
    off, ids = exclusion_csr(ex, 4)
    assert off.dtype == torch.int64 and ids.dtype == torch.int32
    assert off.tolist() == [0, 4, 4, 7, 11]
    assert rows_of(off, ids) == [[3, 3, 7, 12], [], [2, 4, 5], [0, 0, 1, 2 ** 31 - 1]]


@pytest.mark.parametrize("dtype", [torch.int8, torch.int16, torch.int32, torch.int64, torch.uint8])
def test_csr_integer_dtypes(dtype):
    ex = torch.tensor([[9, 1, 5], [2, 2, 0]]).to(dtype)
    off, ids = exclusion_csr(ex, 2)
    assert rows_of(off, ids) == [[1, 5, 9], [0, 2, 2]]


def test_csr_matches_numpy_on_random_rows():
    rng = np.random.Generator(np.random.PCG64(5))
    ex = rng.integers(-20, 1000, size=(300, 40))
    off, ids = exclusion_csr(torch.from_numpy(ex), 300)
    want = [sorted(int(v) for v in r if v >= 0) for r in ex]
    assert rows_of(off, ids) == want


def test_csr_all_padding_and_no_columns_keep_a_valid_ids_array():
    for ex in (torch.full((3, 4), -1), torch.zeros((3, 0), dtype=torch.int64), torch.zeros((0, 5), dtype=torch.int64)):
        Q = ex.shape[0]
        off, ids = exclusion_csr(ex, Q)
        assert off.tolist() == [0] * (Q + 1)
        assert ids.numel() >= 1          # a non-NULL pointer for the kernels even when every row is empty


def test_csr_errors():
    with pytest.raises(ValueError):
        exclusion_csr(torch.zeros(4, dtype=torch.int64), 4)                 # not 2-D
    with pytest.raises(ValueError):
        exclusion_csr(torch.zeros((3, 2), dtype=torch.int64), 4)            # wrong number of rows
    with pytest.raises(ValueError):
        exclusion_csr(torch.zeros((4, 2), dtype=torch.float32), 4)          # not integer ids
    with pytest.raises(ValueError):
        exclusion_csr(torch.zeros((4, 2), dtype=torch.bool), 4)
    with pytest.raises(ValueError):
        exclusion_csr(torch.tensor([[1, 2 ** 31]]), 1)                      # does not fit int32
    with pytest.raises(ValueError):
        exclusion_csr(np.zeros((4, 2), np.int64), 4)                        # not a tensor


def test_null_exclusion_lists_rejected_without_a_gpu():
    lib = _lib.load()
    dummy = 1 << 20     # never dereferenced: the NULL list is rejected first
    off = ids = None
    rc = lib.mr_score_topk_exclude(dummy, dummy, 4, dummy, dummy, 256, 32, 2, 0, 0, dummy, dummy, dummy, 1 << 20,
                                   off, dummy, None)
    assert rc == -1 and b"null" in lib.mr_last_error()
    rc = lib.mr_score_topk_exclude(dummy, dummy, 4, dummy, dummy, 256, 32, 2, 0, 0, dummy, dummy, dummy, 1 << 20,
                                   dummy, ids, None)
    assert rc == -1 and b"null" in lib.mr_last_error()
    rc = lib.mr_topk_rows_exclude(dummy, 4, 256, 256, 2, 0, dummy, dummy, off, dummy, None)
    assert rc == -1 and b"null" in lib.mr_last_error()
    rc = lib.mr_topk_rows_exclude(dummy, 4, 256, 256, 2, 0, dummy, dummy, dummy, ids, None)
    assert rc == -1 and b"null" in lib.mr_last_error()
