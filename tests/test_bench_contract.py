# coding=utf-8
"""bench.py's output contract, checked on the arm that needs no GPU (`--impl reference`: the op-for-op torch-CPU port of the
reference's op sequence on a bounded sample).  One JSON line on stdout, the keys the driver reads, and under torchrun only
rank 0 speaks."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "impl", "cpu_baseline", "e2e")


def _check_line(stdout, n_gpus):
    lines = [l for l in stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "expected exactly one stdout line, got {}: {!r}".format(len(lines), lines[:3])
    rec = json.loads(lines[0])
    for key in REQUIRED:
        assert key in rec, key
    assert rec["impl"] == "reference" and rec["n_gpus"] == n_gpus and rec["steps"] == 1 and rec["warmup"] == 1
    assert rec["unit"] == "edges/s" and rec["higher_is_better"] is True and rec["vs_baseline"] is None
    assert rec["value"] > 0 and rec["ms_per_step"] > 0 and rec["dtype"] == "f32" and rec["data"] == "synthetic"
    assert "workload" in rec["config"] and "model" not in rec["config"]
    cb = rec["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == rec["value"]
    e2e = rec["e2e"]
    assert e2e["value"] == rec["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    return rec


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-sample-div", "400"], cwd=ROOT,
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    _check_line(out.stdout, 1)


def test_reference_arm_under_torchrun_only_rank0_speaks():
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29731", "bench.py", "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "1", "--cpu-sample-div", "400"], cwd=ROOT, capture_output=True, text=True, timeout=900, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    _check_line(out.stdout, 2)


def test_reference_arm_covers_every_baseline_config():
    """--config cfg1..cfg5 on the CPU arm: each BASELINE.json configuration has its own op sequence and declares its sample."""
    for name in ("cfg1", "cfg2", "cfg3", "cfg4", "cfg5"):
        out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--config", name, "--steps", "1", "--warmup", "1",
                              "--cpu-sample-div", "1" if name == "cfg1" else "2000"], cwd=ROOT, capture_output=True, text=True,
                             timeout=600)
        assert out.returncode == 0, (name, out.stderr[-2000:])
        rec = _check_line(out.stdout, 1)
        assert rec["config"]["name"] == name and "reference_sample" in rec["config"]
        assert rec["metric"].startswith("edges/sec")


def test_gpu_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    out = subprocess.run([sys.executable, "bench.py", "--steps", "1", "--warmup", "1"], cwd=ROOT, capture_output=True,
                         text=True, timeout=300)
    assert out.returncode != 0 and out.stdout.strip() == "" and "no CPU fallback" in out.stderr


def test_dump_outputs_samples_large_outputs_to_a_fixed_row_set(tmp_path):
    """Outputs above their share of 64 MB are stored as the same sorted row sample on every call; small ones whole."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    big = torch.arange(200000, dtype=torch.float32)[:, None].repeat(1, 128)      # each row holds its own index
    small = torch.randn(1000, 16)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), ("big", "small"), (big, small))
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64 * 1000 * 1000
    got = np.load(tmp_path / "a" / "big.npy")
    assert got.dtype == np.float32 and got.shape[1] == 128 and 0 < got.shape[0] < 200000
    rows = got[:, 0].astype(np.int64)
    assert np.all(np.diff(rows) > 0) and np.array_equal(got, big.numpy()[rows])
    assert np.array_equal(got, np.load(tmp_path / "b" / "big.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small.numpy())


@pytest.mark.gpu
def test_gpu_arm_dumps_the_outputs_of_its_last_step(tmp_path):
    """--dump-outputs on the headline step: one float32 file per layer, within 64 MB, the same arrays on a second run."""
    import numpy as np
    dumps = []
    for run in ("first", "second"):
        out = subprocess.run([sys.executable, "bench.py", "--steps", "2", "--warmup", "1", "--scale", "0.1", "--no-cpu-baseline",
                              "--no-e2e", "--dump-outputs", str(tmp_path / run)], cwd=ROOT, capture_output=True, text=True,
                             timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout)["steps"] == 2
        assert sorted(os.listdir(tmp_path / run)) == ["gat.npy", "gcn.npy"]
        assert sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= 64 * 1000 * 1000
        dumps.append({f: np.load(tmp_path / run / f) for f in ("gat.npy", "gcn.npy")})
    for f, a in dumps[0].items():
        assert a.dtype == np.float32 and a.shape[1] == 128 and np.all(np.isfinite(a)) and np.any(a != 0), f
        assert np.array_equal(a, dumps[1][f]), f
