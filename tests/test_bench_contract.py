"""The driver's bench.py contract: one JSON line on stdout with the agreed keys."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _last_json(stdout: str) -> dict:
    lines = [ln for ln in stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1, stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_reports_unavailable():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "3"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = _last_json(r.stdout)
    assert line["impl"] == "reference" and isinstance(line["unavailable"], str) and len(line["unavailable"]) > 10


@pytest.mark.gpu
def test_bench_line_on_a_tiny_model():
    """Same code path as the headline run (GRPO, native sampler, DeBERTa reward, graph micro-steps, pinned H2D / D2H) at toy size."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--model", "tiny", "--reward", "deberta-tiny", "--response-length", "48",
                        "--mini-batches", "1", "--steps", "2", "--warmup", "3"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = _last_json(r.stdout)
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "e2e", "gpu_launches", "clocks"):
        assert k in line, k
    assert line["metric"] == "episodes_per_sec" and line["n_gpus"] == 1 and line["steps"] == 2 and line["warmup"] == 3
    assert line["value"] > 0 and line["higher_is_better"] is True and line["scaling"] == "weak" and line["dtype"] == "bf16"
    assert abs(line["value"] * line["ms_per_step"] / 1e3 - line["config"]["global_batch"]) < 1e-6 * line["config"]["global_batch"] + 1e-3
    assert line["e2e"]["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    assert line["e2e"]["value"] <= line["value"] * 1.001          # wall clock around the same steps cannot beat the device time
    assert line["gpu_launches"] > 100
    assert set(line["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_update(tmp_path):
    """``--dump-outputs``: after exactly ``--steps`` timed updates, the last one's rollout, metrics and a weight sample land in
    float32 / float64 ``.npy`` files of at most 64 MB in all."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--model", "tiny", "--reward", "deberta-tiny", "--response-length", "48",
                        "--mini-batches", "1", "--steps", "2", "--warmup", "1", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = _last_json(r.stdout)
    assert len([ln for ln in r.stderr.splitlines() if ln.startswith("[bench] step ")]) == 2 and line["steps"] == 2
    arrays = {f[:-len(".npy")]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64e6
    rows = arrays["responses"].shape[0]
    assert rows > 0 and arrays["responses"].shape == (rows, 48)
    for k in ("logprobs", "ref_logprobs", "advantages"):
        assert arrays[k].shape == (rows, 48) and np.isfinite(arrays[k]).all(), k
    assert arrays["scores"].shape == arrays["normalized_scores"].shape == (rows,)
    assert (arrays["responses"] == np.round(arrays["responses"])).all() and (arrays["responses"] >= 0).all()
    assert arrays["trainable_weights_sample"].size > 0 and np.isfinite(arrays["trainable_weights_sample"]).all()
    assert {"metrics.loss.policy_avg_new", "metrics.objective.kl_old"} <= set(arrays)
    assert not any(k.startswith(("metrics.time.", "metrics.throughput.")) for k in arrays)
