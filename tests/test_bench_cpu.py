"""Control-flow dry runs of the headline benchmark (``bench.py --device cpu``: gloo, PyTorch engine, host timers).
The numbers are meaningless; what is checked is that every phase of the script (warm-up, device-timed loop, pipelined
end-to-end loop with H2D of q/k/v/dO and a D2H result per step, the compute-only communication probe, the max-over-
ranks reductions) runs to completion and that the ONE JSON line carries the keys of the driver's contract."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches"}


def _run(n, port, *flags):
    cmd = [sys.executable]
    if n > 1:
        cmd += ["-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
                "--master-port", str(port)]
    cmd += [os.path.join(ROOT, "bench.py"), "--gpus", str(n), "--steps", "2", "--warmup", "1", "--device", "cpu",
            "--seq", "256", "--heads", "4", "--head-dim", "16", *flags]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


def test_bench_single_process_contract():
    d = _run(1, 0)
    assert KEYS <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] >= 3 and d["higher_is_better"] is True
    assert d["metric"] == "attention_tflops_fwd_bwd" and d["config"]["seq_len"] == 256
    e = d["e2e"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(e)
    assert e["h2d_bytes_per_step"] == 4 * 256 * 4 * 16 * 2          # q, k, v and dO shards in bf16
    assert e["d2h_bytes_per_step"] == 4 and d["ms_per_step"] > 0 and e["ms_per_step"] > 0


def test_bench_dump_outputs_repeat_exactly(tmp_path):
    """``--dump-outputs``: out / dq / dk / dv of the last timed step as float32, identical for identical inputs (the
    gradients are that step's alone, whatever the number of steps)."""
    import numpy as np
    dumps = []
    for run, steps in (("a", "2"), ("b", "3")):
        d = _run(1, 0, "--steps", steps, "--dump-outputs", str(tmp_path / run))
        assert d["steps"] == int(steps)
        assert d["outputs"]["arrays"] == ["out", "dq", "dk", "dv"] and d["outputs"]["rows_per_rank"] == 256
        dumps.append({n: np.load(tmp_path / run / f"{n}.npy") for n in d["outputs"]["arrays"]})
    for n, x in dumps[0].items():
        assert x.dtype == np.float32 and x.shape == (1, 1, 256, 4, 16) and np.isfinite(x).all()
        assert np.array_equal(x, dumps[1][n]), n
    assert np.abs(dumps[0]["dq"]).max() > 0


def test_bench_dump_outputs_two_ranks_forward(tmp_path):
    d = _run(2, 29861, "--mode", "fwd", "--dump-outputs", str(tmp_path))
    import numpy as np
    out = np.load(tmp_path / "out.npy")
    assert d["outputs"]["arrays"] == ["out"] and out.shape == (2, 1, 128, 4, 16) and out.dtype == np.float32
    assert sorted(os.listdir(tmp_path)) == ["out.npy"]


def test_dump_outputs_samples_rows_within_budget(tmp_path):
    import importlib.util

    import numpy as np
    import torch
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    x = torch.randn(2, 1000, 3, 8, dtype=torch.bfloat16)
    y = torch.randn(2, 1000, 1, 8)
    budget = 40_000
    info = bench.dump_outputs(str(tmp_path), {"x": x, "y": y}, None, 0, budget=budget)
    n = info["rows_per_rank"]
    assert 0 < n < 1000 and info["row_sample_seed"] == 0
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= budget
    xs, ys = np.load(tmp_path / "x.npy"), np.load(tmp_path / "y.npy")
    assert xs.shape == (1, 2, n, 3, 8) and ys.shape == (1, 2, n, 1, 8)
    rows = torch.randperm(1000, generator=torch.Generator().manual_seed(0))[:n].sort().values
    assert np.array_equal(xs[0], x[:, rows].float().numpy()) and np.array_equal(ys[0], y[:, rows].numpy())
    again = bench.dump_outputs(str(tmp_path / "again"), {"x": x, "y": y}, None, 0, budget=budget)
    assert again == {**info, "dir": str(tmp_path / "again")}


@pytest.mark.parametrize("flags", [
    (),
    ("--mode", "fwd", "--ring-impl", "strip"),
    ("--ulysses", "2", "--window", "64", "--kv-heads", "2"),
    ("--ulysses", "2", "--qkvpacked", "--ring-impl", "basic"),
])
def test_bench_two_ranks_all_phases(flags):
    d = _run(2, 29871 + len(flags), *flags)
    assert KEYS <= set(d) and d["n_gpus"] == 2
    assert d["e2e"]["h2d_bytes_per_step"] > 0
    comm = d["comm"]
    assert comm is not None and "error" not in comm, comm
    assert comm["compute_only_ms"] > 0 and "exposed_comm_ms" in comm


def test_bench_multi_config_in_one_process_group():
    """``--configs 2,3 --modes fwd,fwdbwd``: one JSON line per config x mode from ONE launch (the presets' shapes are
    overridden by explicit flags, so the dry run stays tiny)."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29741", os.path.join(ROOT, "bench.py"), "--gpus", "2", "--steps", "1", "--warmup", "1",
           "--device", "cpu", "--seq", "128", "--heads", "4", "--head-dim", "16", "--configs", "2,3", "--modes", "fwd,fwdbwd",
           "--no-comm-probe"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]
    assert [(d["config_id"], d["config"]["mode"]) for d in lines] == [(2, "fwd"), (2, "fwdbwd"), (3, "fwd"), (3, "fwdbwd")]
    assert lines[0]["config"]["parallelism"] == "ulysses2xring1" and lines[2]["config"]["parallelism"] == "ulysses1xring2"
