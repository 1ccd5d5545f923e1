"""bench.py contract (CPU part): the reference arm prints exactly one JSON line with the keys the driver reads, for both
workloads.  (The CUDA arm is exercised on the GPU box by the driver itself.)"""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

REQUIRED = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"}


@pytest.mark.parametrize("workload", ["muzero", "efficientzero"])
def test_reference_arm_prints_one_json_line(workload):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", workload, "--steps", "1",
                          "--warmup", "0", "--cpu-sample-roots", "8", "--sims", "4"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert REQUIRED <= set(d), REQUIRED - set(d)
    assert d["impl"] == "reference" and d["unit"] == "simulations/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert "workload" in d["config"] and ("EfficientZero" in d["config"]["workload"]) == (workload == "efficientzero")


def test_dump_outputs_writes_float32_and_samples_past_the_limit(tmp_path, monkeypatch):
    """--dump-outputs: one float32 .npy per returned array; past the size limit, the same seeded rows of every array."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    g = torch.Generator().manual_seed(0)
    result = dict(visits=torch.randint(0, 50, (512, 6), dtype=torch.int32, generator=g), values=torch.rand(512, generator=g),
                  nlegal=torch.full((512,), 6, dtype=torch.int32), policy_logits=torch.randn(512, 6, generator=g))
    bench.dump_outputs(str(tmp_path / "all"), result)
    for k, v in result.items():
        a = np.load(tmp_path / "all" / f"{k}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, v.numpy().astype(np.float32))
    assert not (tmp_path / "all" / "rows.npy").exists()

    monkeypatch.setattr(bench, "DUMP_LIMIT", 4096 + 20 * (14 * 4 + 8))      # room for 20 of the 512 roots
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), result)
    rows = np.load(tmp_path / "s1" / "rows.npy")
    assert rows.dtype == np.float64 and len(rows) == 20 and np.array_equal(rows, np.load(tmp_path / "s2" / "rows.npy"))
    idx = rows.astype(np.int64)
    for k, v in result.items():
        assert np.array_equal(np.load(tmp_path / "s1" / f"{k}.npy"), v.numpy()[idx].astype(np.float32))
    assert sum(f.stat().st_size for f in (tmp_path / "s1").iterdir()) <= bench.DUMP_LIMIT
