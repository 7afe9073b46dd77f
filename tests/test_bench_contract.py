"""CPU: the reference arm of bench.py prints exactly one JSON line with the contract's keys (the GPU arm needs a
device; its line carries the same keys plus `roofline`, `clocks`, `gpu_launches`)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, f"stdout must hold exactly one JSON line, got {len(lines)}"
    return json.loads(lines[0])


def test_reference_arm_json_contract():
    line = run("--impl", "reference", "--workload", "cfg1", "--steps", "2", "--warmup", "1")
    assert line["steps"] == 2 and line["warmup"] == 1
    assert line["impl"] == "reference"
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["vs_baseline"] is None and line["data"] == "synthetic" and "workload" in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["value"] > 0 and line["higher_is_better"] is True


def test_reference_arm_other_ranks_print_nothing():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--workload", "cfg1", "--steps", "1", "--warmup", "0"], capture_output=True, text=True,
                         timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_arm_falls_back_to_the_port_without_the_installed_reference(tmp_path, monkeypatch):
    """Without baseline/_ref the CPU arm is the oracle port and says so."""
    import importlib
    sys.path.insert(0, ROOT)
    bw = importlib.import_module("bench_workloads")
    monkeypatch.setattr(bw, "reference_package", lambda: None)
    wl = bw.WORKLOADS["cfg1"](0, 1, None)
    res = wl.reference_arm(steps=1, warmup=0)
    assert res["kind"] == "port" and res["value"] > 0 and res["ms_per_step"] > 0


def test_dump_outputs_writes_float_arrays_within_the_limit(tmp_path):
    import importlib
    sys.path.insert(0, ROOT)
    bench = importlib.import_module("bench")
    out = {"merged": np.arange(5, dtype=np.float32), "NDCG@10": np.float64(0.25)}
    bench.dump_outputs(str(tmp_path / "d"), out)
    assert sorted(os.listdir(tmp_path / "d")) == ["NDCG@10.npy", "merged.npy"]
    assert np.array_equal(np.load(tmp_path / "d" / "merged.npy"), out["merged"])
    assert np.load(tmp_path / "d" / "NDCG@10.npy") == 0.25
    with pytest.raises(TypeError):
        bench.dump_outputs(str(tmp_path / "ints"), {"ids": np.arange(3)})
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_LIMIT_BYTES // 4 + 1, np.float32)})
    assert not (tmp_path / "ints").exists() and not (tmp_path / "big").exists()


def test_large_outputs_are_a_fixed_sample():
    import importlib
    import torch
    sys.path.insert(0, ROOT)
    bw = importlib.import_module("bench_workloads")
    t = torch.arange(bw.OUTPUT_SAMPLE + 1000, dtype=torch.float64)
    a, b = bw._output(t), bw._output(t)
    assert a.dtype == np.float32 and a.shape == (bw.OUTPUT_SAMPLE,)
    assert np.array_equal(a, b) and np.all(np.diff(a) > 0)
    small = torch.ones(3, 4)
    assert bw._output(small).shape == (3, 4)


def test_bench_rejects_zero_steps():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


@pytest.mark.gpu
def test_dumped_outputs_repeat_from_run_to_run(tmp_path):
    """Same arguments, same seeded inputs: two runs dump the same arrays (the headline metrics and the companion merge)."""
    env = dict(os.environ, MR_BENCH_SKIP_ACCURACY="1")
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1", "--steps", "2",
                              "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
        assert out.returncode == 0, out.stderr[-2000:]
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["NDCG@10.npy", "Recall@10.npy", "merger.merged.npy"]
    assert names == sorted(os.listdir(tmp_path / "b"))
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), n


def test_configs_do_not_depend_on_the_run():
    """`config` must be identical in the GPU arm and the reference arm: a pure function of the workload definition."""
    import importlib
    sys.path.insert(0, ROOT)
    bw = importlib.import_module("bench_workloads")
    for name, cls in bw.WORKLOADS.items():
        assert cls(0, 1, None).config() == cls(3, 8, None).config(), name
        assert "workload" in cls(0, 1, None).config()
    assert bw.DEFAULT_WORKLOAD == "eval_cfg5"
