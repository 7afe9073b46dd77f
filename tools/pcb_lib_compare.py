"""get_pcb_vectors at K = 8 BLaIR-base (seeded inputs): another build of libmergerec_b200.so (e.g. the parent commit's)
against this tree's, in one process -- output checksums of both, device times alternated between the two builds --
plus the single-GPU get_pcb_vectors + merge and get_pcb_vectors_sharded on one GPU.  One JSON line on stdout.

    python tools/pcb_lib_compare.py /path/to/other/libmergerec_b200.so"""
import ctypes
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mergerec_b200 import _lib, synth  # noqa: E402
from mergerec_b200.merger.algorithms._common import merge_axpy, weights_tensor  # noqa: E402
from mergerec_b200.merger.algorithms.pcb import get_pcb_vectors  # noqa: E402
from mergerec_b200.merger.sharded import get_pcb_vectors_sharded  # noqa: E402

new = _lib.load()
par = ctypes.CDLL(os.path.abspath(sys.argv[1]))
for name, (a, r) in _lib.SIGNATURES.items():
    if hasattr(par, name):
        f = getattr(par, name)
        f.argtypes, f.restype = a, r
d, K = synth.total_numel(synth.roberta_shapes()), 8
g = torch.Generator(device="cuda").manual_seed(1234)
base = torch.randn(d, generator=g, device="cuda") * 0.02
models = [base + 1e-3 * torch.randn(d, generator=g, device="cuda") for _ in range(K)]


def chk(t):
    return int(t.contiguous().view(torch.int32).to(torch.int64).sum())


def timed(fn, iters=10):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


res = {"d": d, "K": K}
for nm, lib in (("other", par), ("new", new)):
    _lib._lib = lib
    res[f"vectors_checksum_{nm}"] = chk(get_pcb_vectors(base, models, density=0.2)[:, :d])
times = {"other": [], "new": []}
for rep in range(6):
    for nm, lib in (("other", par), ("new", new)) if rep % 2 == 0 else (("new", new), ("other", par)):
        _lib._lib = lib
        times[nm].append(timed(lambda: get_pcb_vectors(base, models, density=0.2)))
res["get_pcb_vectors_ms"] = times
_lib._lib = new
w = weights_tensor([0.3] * K, "cuda")
out = torch.empty(d, device="cuda")


def single():
    v = get_pcb_vectors(base, models, density=0.2)
    merge_axpy(base, list(v.unbind(0)), w, _lib.MR_ORDER_BASE_FIRST, False, out=out)


res["single_gpu_pcb_plus_merge_ms"] = [timed(single) for _ in range(3)]
res["merged_bits_checksum_single_gpu"] = chk(out)
res["sharded_world1_vectors_ms"] = [timed(lambda: get_pcb_vectors_sharded(base, models, 0.2, d)) for _ in range(3)]
res["sharded_world1_equal"] = bool(torch.equal(get_pcb_vectors_sharded(base, models, 0.2, d)[:, :d].contiguous().view(torch.int32),
                                               get_pcb_vectors(base, models, density=0.2)[:, :d].contiguous().view(torch.int32)))
print(json.dumps(res))
