"""bench.py's driver contract, checked on the CPU: the reference arm prints exactly one JSON line with the agreed keys
(stdout carries nothing else), non-zero ranks of a reference run exit without work, and the product arm refuses to run
without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

import oracle_lib as ol

ROOT = ol.ROOT
SMALL = ["--docs", "20000", "--vocab", "2000", "--dim", "128", "--batch", "64", "--steps", "2", "--warmup", "1", "--cpu-sample", "32"]


def run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, cwd=ROOT, env=e, timeout=600)


def test_reference_arm_prints_one_json_line():
    r = run(["--impl", "reference"] + SMALL)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "queries/sec" and d["unit"] == "queries/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0
    assert d["config"]["workload"] == "hybrid10m" and d["config"]["batch"] == 64
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    r = run(["--impl", "reference"] + SMALL, env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_needs_cuda():
    import torch
    if torch.cuda.is_available():
        return
    r = run(SMALL)
    assert r.returncode != 0 and r.stdout.strip() == ""
    assert "no CPU fallback" in r.stderr


def _dumped(d):
    import numpy as np
    files = sorted(os.listdir(d))
    arrays = {f: np.load(os.path.join(d, f)) for f in files}
    assert "count.npy" in arrays and "key.npy" in arrays
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(os.path.getsize(os.path.join(d, f)) for f in files) <= 64 << 20
    return arrays


def _same_outputs(args, n_queries, tmp_path):
    import numpy as np
    runs = []
    for i in range(2):
        r = run(args + ["--dump-outputs", str(tmp_path / str(i))])
        assert r.returncode == 0, r.stderr[-2000:]
        runs.append(_dumped(tmp_path / str(i)))
    assert runs[0].keys() == runs[1].keys()
    for f in runs[0]:
        assert np.array_equal(runs[0][f], runs[1][f]), f
    n = runs[0]["count.npy"]
    assert len(n) == n_queries and n.sum() > 0 and (runs[0]["key.npy"][:, :int(n.max())] != 0).any()


def test_reference_arm_dumps_the_same_outputs_every_run(tmp_path):
    _same_outputs(["--impl", "reference"] + SMALL, 32, tmp_path)


@pytest.mark.gpu
def test_product_arm_dumps_the_same_outputs_every_run(tmp_path):
    _same_outputs(SMALL + ["--no-cpu-baseline", "--no-other-configs", "--no-graph-cache", "--recall-queries", "0"], 64, tmp_path)
