"""CPU: argument handling of the sharded PCB / DARE merges.  `ShardedModelMerger.merge("pcb" | "dare")` rejects bad
weights, a missing base model, a bad DARE density and a wrong mask shape with the exceptions `ModelMerger.merge`
raises, before any kernel runs; the C entry points of the sharded PCB search (mr_pcb_vectors_dist and its host-only
plan query) reject bad arguments with a negative status and a message without touching a device."""
import ctypes as C

import pytest
import torch

from mergerec_b200 import _lib
from mergerec_b200.merger import ModelMerger
from mergerec_b200.merger.sharded import ShardedModelMerger


def _bare(cls, K=3, d=70, base=True):
    """A merger holding CPU flat vectors, built without the constructor (which needs a GPU to flatten)."""
    m = object.__new__(cls)
    m.models = [torch.zeros(d) for _ in range(K)]
    m.base_model = torch.zeros(d) if base else None
    m.shape_dict = {"w": torch.Size([d])}
    if cls is ShardedModelMerger:
        m.group, m.d_global, m.bounds = None, d, (0, d)
    return m


@pytest.mark.parametrize("merge_type", ["pcb", "dare"])
def test_bad_weights_and_missing_base_raise_like_model_merger(merge_type):
    for cls in (ModelMerger, ShardedModelMerger):
        with pytest.raises(ValueError, match="Weights should be a float or a list of floats"):
            _bare(cls).merge(merge_type, [1, 2, 3], density=0.2)
        with pytest.raises(ValueError, match="Weights should be a float or a list of floats"):
            _bare(cls).merge(merge_type, "0.3", density=0.2)
        name = "PCB" if merge_type == "pcb" else "DARE"
        with pytest.raises(ValueError, match=f"{name} merge requires a base model"):
            _bare(cls, base=False).merge(merge_type, 0.3, density=0.2)


@pytest.mark.parametrize("density", [-0.1, 1.5])
def test_bad_dare_density_raises_like_model_merger(density):
    for cls in (ModelMerger, ShardedModelMerger):
        with pytest.raises(ValueError, match="dropout probability has to be between 0 and 1"):
            _bare(cls).merge("dare", 0.3, density=density)


def test_missing_dare_density_raises_like_model_merger():
    for cls in (ModelMerger, ShardedModelMerger):
        with pytest.raises(TypeError):
            _bare(cls).merge("dare", 0.3)


def test_wrong_mask_shape_and_model_count():
    m = _bare(ShardedModelMerger, K=3, d=70)
    for shape in ((3, 69), (2, 70), (70,)):
        with pytest.raises(ValueError, match="masks must have shape"):
            m.merge("dare", 0.3, density=0.1, masks=torch.ones(shape, dtype=torch.bool))
    for mt, kw in (("pcb", dict(density=0.2)), ("dare", dict(density=0.1))):
        with pytest.raises(AssertionError, match="Number of models and weights should match"):
            m.merge(mt, [0.1, 0.2], **kw)


def test_unknown_merge_type_still_raises():
    with pytest.raises(ValueError, match="is not supported"):
        _bare(ShardedModelMerger).merge("pcb_v2", 0.3)


# ---------------------------------------------------------------------------------------------------------- C ABI
FAKE = C.c_void_p(256)          # never dereferenced: every call below fails its argument checks first


def _call(d_local=64, j_off=0, d_global=128, K=2, q_index=10, phase=0, flags=0, base=FAKE, models="fake", lo=FAKE,
          hi=FAKE, status=FAKE, out=FAKE, ldo=64, ws=FAKE, ws_bytes=1 << 40):
    lib = _lib.load()
    if models == "fake":
        models = (C.c_void_p * K)(*([256] * K))
    rc = lib.mr_pcb_vectors_dist(base, models, K, d_local, j_off, d_global, lo, hi, q_index, flags, phase, status, out, ldo,
                                 ws, ws_bytes, None)
    return rc, lib.mr_last_error().decode()


def test_dist_entry_point_rejects_bad_arguments():
    cases = [
        (dict(j_off=16), "multiple of 32"),                               # misaligned slice start
        (dict(j_off=96, d_local=64), "j_off + d_local <= d_global"),     # slice past the end
        (dict(d_local=-1), "0 <= d_local"),
        (dict(d_local=40), "multiple of 32 columns or at d_global"),     # a ragged slice that is not the last one
        (dict(phase=-1), "phase -1 outside"),
        (dict(phase=4), "phase 4 outside [0,4)"),                        # d_global = 128: the dense search has 4 phases
        (dict(d_global=1 << 20, d_local=1 << 19, ldo=1 << 19, phase=7), "phase 7 outside [0,7)"),   # fast search: 7
        (dict(q_index=128), "quantile index"),
        (dict(K=0), "K=0"),
        (dict(K=17), "K=17"),
        (dict(d_global=1 << 32, d_local=64), "d_global"),
        (dict(lo=None), "null pointer"),
        (dict(hi=None), "null pointer"),
        (dict(status=None), "null pointer"),
        (dict(ws=None), "null pointer"),
        (dict(base=None), "null pointer"),
        (dict(models=None), "null pointer"),
        (dict(out=None), "null pointer"),
        (dict(models=(C.c_void_p * 2)(256, 0)), "models[1] is NULL"),
        (dict(ldo=32), "ldo >= d_local"),
    ]
    for kw, msg in cases:
        rc, err = _call(**kw)
        assert rc == -1 and msg in err, (kw, rc, err)


def test_dist_plan_is_a_host_query():
    lib = _lib.load()
    plan = (C.c_int32 * 8)()
    S, M = _lib.MR_PCB_SUM, _lib.MR_PCB_MAX
    # fast search from d_global = 1024 * 128 on (the sample of one quad per 128 columns holds >= 4096 elements)
    assert lib.mr_pcb_dist_plan(1024 * 128, 0, plan, 8) == 7
    assert list(plan)[:7] == [S, S, S, S | M, S, S, 0]
    assert lib.mr_pcb_dist_plan(1024 * 128 - 1, 0, plan, 8) == 4
    assert list(plan)[:4] == [S | M, S, S, 0]
    assert lib.mr_pcb_dist_plan(1 << 30, _lib.MR_PCB_DENSE | _lib.MR_PCB_IEEE, plan, 8) == 4
    assert lib.mr_pcb_dist_plan(1 << 30, _lib.MR_PCB_IEEE, None, 0) == 7
    assert lib.mr_pcb_dist_plan(0, 0, plan, 8) == -1 and b"d_global" in lib.mr_last_error()
    assert lib.mr_pcb_dist_plan(100, 0, None, 4) == -1 and b"null" in lib.mr_last_error()
