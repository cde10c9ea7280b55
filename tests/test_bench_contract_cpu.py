"""bench.py contract on the CPU arm (no GPU needed): `--impl reference` prints ONE JSON line on stdout with the keys the
driver reads, times the oracle port on host threads, and the B200 arm refuses to run without a CUDA device."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def test_reference_arm_json_line():
    res = _run(["--impl", "reference", "--config", "2", "--steps", "1", "--warmup", "0"])
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1                                   # stdout carries only the JSON line
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "davidson_sigma_vectors_per_s" and d["unit"] == "sigma-vectors/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["config"]["workload"].startswith("cfg2") and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0


def test_step_counts_and_dump_flag_are_checked():
    for args in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "unused"]):
        res = _run(args, timeout=120)
        assert res.returncode == 2 and "error:" in res.stderr, args


def test_dump_sample_is_seeded_and_bounded():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    a = np.arange(3 * 1000, dtype=np.float64).reshape(3, 1000)
    kept, cols = bench.sample_columns(a, a.nbytes)
    assert kept is a and cols is None
    kept, cols = bench.sample_columns(a, 3 * 8 * 100 + 7)
    assert kept.shape == (3, 100) and kept.nbytes <= 3 * 8 * 100 + 7
    assert np.all(np.diff(cols) > 0) and np.array_equal(kept, a[:, cols])
    again, cols2 = bench.sample_columns(a, 3 * 8 * 100 + 7)
    assert np.array_equal(cols, cols2) and np.array_equal(kept, again)


def test_b200_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        return                                               # on a GPU box the arm runs; covered by the bench itself
    res = _run(["--config", "1", "--steps", "1", "--warmup", "0", "--davidson", "0", "--no-cpu-baseline"])
    assert res.returncode != 0
    assert "no CPU fallback" in res.stderr or "needs a B200" in res.stderr
