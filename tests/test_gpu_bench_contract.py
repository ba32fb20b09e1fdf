"""bench.py's own arm on a small batch: one JSON line on stdout with every key of the measurement contract."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu


def test_bench_prints_contract_line():
    r = subprocess.run([sys.executable, os.path.join(util.ROOT, "bench.py"), "--envs", "512", "--steps", "12", "--warmup", "3",
                        "--burn-in", "20", "--no-cpu-baseline"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[:500]
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline"):
        assert k in d, k
    assert d["metric"] == "env-steps/sec" and d["steps"] == 12 and d["n_gpus"] == 1 and d["dtype"] == "f64"
    # NoMove + scripted gaze: the K steps of a replica are ONE d2d_rollout launch; the per-step-launch figure rides along
    assert d["gpu_launches"] == 1 and d["value"] > 0 and d["vs_baseline"] is None and d["scaling"] == "weak"
    ssl = d["single_step_launches"]
    assert ssl["gpu_launches"] == 12 and ssl["value"] > 0 and abs(ssl["value"] - 512 / (ssl["ms_per_step"] * 1e-3)) <= 1e-6 * ssl["value"]
    assert abs(d["value"] - 512 / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]
    assert d["method"]["replicas"] >= 2 and "workload" in d["config"] and "l2" in d["config"]   # a small batch needs replicas to stay L2-cold
    # the timed region is exactly --steps steps of every env: one replay of a graph holding K steps of every replica
    assert d["method"]["timed_steps_per_env"] == 12 and d["method"]["graph_replays"] == 1
    assert abs(d["method"]["timed_region_ms_this_rank"] - d["ms_per_step"] * 12 * d["method"]["replicas"]) < 1e-9
    assert d["per_step_events"]["steps"] == 12 and d["e2e"]["steps"] == 12
    assert len(d["per_rank"]) == 1 and abs(d["per_rank"][0]["ms_per_step"] - d["ms_per_step"]) < 1e-12
    assert "workloads" not in d                                              # only the default (config 2, full size) run carries them
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 512 * 8 and e["d2h_bytes_per_step"] > 0
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-12
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}


def _bench_dump(d, steps):
    r = subprocess.run([sys.executable, os.path.join(util.ROOT, "bench.py"), "--envs", "256", "--steps", str(steps), "--warmup", "3",
                        "--burn-in", "0", "--no-cpu-baseline", "--dump-outputs", str(d)],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert sum(f.stat().st_size for f in d.glob("*.npy")) <= 64 << 20
    return json.loads(r.stdout), {f.stem: np.load(f) for f in sorted(d.glob("*.npy"))}


def test_bench_dump_outputs_are_the_timed_steps(tmp_path):
    """--dump-outputs holds float32 / float64 arrays of the timed envs after their last timed step, identical from run to run
    with the same arguments.  The NoMove + scripted-gaze workload reaches its last timed step after W eager warm-up steps,
    the burn-in (0 here), a W-step d2d_rollout warm-up call and the K timed steps, so an env whose episode has not ended
    reports exactly 2 W + K steps."""
    j, a = _bench_dump(tmp_path / "a", 7)
    _, b = _bench_dump(tmp_path / "b", 7)
    _, c = _bench_dump(tmp_path / "c", 8)
    rows = j["method"]["replicas"] * 256
    assert {"local_map", "yaw_angle", "done", "belief", "steps", "env_index"} <= set(a) and set(a) == set(b) == set(c)
    idx = a["env_index"]
    assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < rows and np.array_equal(idx, np.round(idx))
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and a[k].shape[0] == len(idx), k
        assert np.array_equal(a[k], b[k]), k
    for dump, k in ((a, 7), (c, 8)):
        steps = dump["steps"]
        assert steps.max() == 2 * 3 + k and np.mean(steps == 2 * 3 + k) > 0.5, (k, np.unique(steps))
