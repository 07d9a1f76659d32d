"""bench.py's contract: the reference arm (the oracle port on the host cores) prints one JSON line with the agreed keys, the
GPU arm refuses to run without a device instead of falling back, and ``--dump-outputs`` writes what the timed path
computed."""
import json
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*flags):
    return subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), *flags], cwd=REPO, capture_output=True,
                          text=True, timeout=600)


def test_reference_arm_line():
    proc = _run("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert proc.returncode == 0, proc.stderr[-2000:]
    line = json.loads(proc.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["unit"] == "instances/s"
    assert line["n_gpus"] == 1 and line["steps"] == 1 and line["warmup"] == 0 and line["value"] > 0
    base = line["cpu_baseline"]
    assert base["kind"] == "port" and base["cores"] >= 1 and base["value"] == line["value"] and base["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    baseline = json.load(open(os.path.join(REPO, "BASELINE.json")))
    assert line["metric"] == baseline["metric"]


def test_dump_outputs_is_refused_by_the_reference_arm(tmp_path):
    proc = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path / "out"))
    assert proc.returncode == 2 and "--dump-outputs" in proc.stderr
    assert not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_step(tmp_path):
    """The dumped phi is what the timed device path computed: two classes of opposite sign, and per instance the
    components add up to logit f(x) - logit E[f(background)] (the logit link's efficiency property)."""
    import numpy as np
    from distributedkernelshap_b200.datasets import adult_like
    proc = _run("--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-other-mode", "--no-other-configs",
                "--dump-outputs", str(tmp_path))
    assert proc.returncode == 0, proc.stderr[-2000:]
    line = json.loads(proc.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["warmup"] == 1
    phi = np.load(tmp_path / "shap_values.npy")
    assert [p.name for p in tmp_path.iterdir()] == ["shap_values.npy"]
    assert phi.dtype == np.float64 and phi.shape == (2, 2560, 12) and np.isfinite(phi).all()
    np.testing.assert_allclose(phi[0], -phi[1], rtol=0, atol=1e-12)
    d = adult_like(n_explain=2560, n_background=100, seed=0)
    fx = d["predictor"].predict_proba(d["X_explain"])[:, 1]
    f0 = d["predictor"].predict_proba(d["background"])[:, 1].mean()
    np.testing.assert_allclose(phi[1].sum(1) + np.log(f0 / (1 - f0)), np.log(fx / (1 - fx)), rtol=1e-7, atol=1e-7)


def test_gpu_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    proc = _run("--steps", "1", "--warmup", "0", "--no-cpu-baseline")
    assert proc.returncode != 0
    assert "no CPU fallback" in (proc.stdout + proc.stderr)
