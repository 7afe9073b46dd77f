"""`Evaluator.label_log_softmax` over NCCL on a sharded item table: needs at least two GPUs, skipped otherwise.

Either launch pytest itself under torchrun (`WORLD_SIZE > 1`: every rank runs the worker in-process), or run plain pytest
on a box with >= 2 GPUs: the test then starts `torch.distributed.run --nproc-per-node <min(#GPUs, 8)>` on
tests/nccl_label_log_softmax_worker.py.  On one GPU, tests/test_label_log_softmax_gpu.py plays the same exchange by hand."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_sharded_label_log_softmax_over_nccl():
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import nccl_label_log_softmax_worker
        assert nccl_label_log_softmax_worker.main() == 0
        return
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (or a torchrun launch with WORLD_SIZE > 1)")
    n = min(n, 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(HERE, "nccl_label_log_softmax_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, (out.stdout[-2000:], out.stderr[-4000:])
    assert "nccl label-log-softmax worker: ok" in out.stdout
