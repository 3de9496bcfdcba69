"""bench.py prints exactly one strict-JSON line with the keys the driver reads.  The reference arm runs on the CPU
(a tiny sample here); the GPU arm is exercised under -m gpu."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def _one_json_line(stdout):
    lines = [ln for ln in stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0], parse_constant=lambda c: (_ for _ in ()).throw(ValueError(f"non-finite {c}")))


def test_reference_arm_line():
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "4", "--warmup", "3",
                          "--cpu-steps-per-proc", "8"], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = _one_json_line(out.stdout)
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["value"] > 0 and d["unit"] == "env-steps/s"
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["config"]["workload"] and d["higher_is_better"] is True and d["vs_baseline"] is None


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "2"], cwd=ROOT,
                         capture_output=True, text=True, env=env, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_types_and_cap(tmp_path, monkeypatch):
    import numpy as np
    import bench
    rng = np.random.default_rng(0)
    arrays = {"obs": rng.normal(size=(100, 137)).astype(np.float32), "reward": rng.normal(size=100),
              "flags": rng.integers(0, 4, size=100, dtype=np.uint8)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    got = {k: np.load(tmp_path / "all" / f"{k}.npy") for k in ("obs", "reward", "flags")}
    assert not (tmp_path / "all" / "env_index.npy").exists()
    assert got["obs"].dtype == np.float32 and got["reward"].dtype == np.float64 and got["flags"].dtype == np.float32
    for k in arrays:
        assert np.array_equal(got[k], arrays[k])
    # over the cap: the same seeded rows of every array, and their indices
    monkeypatch.setattr(bench, "DUMP_BYTES_MAX", 30 * 1024 + 4096 * 4)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["env_index.npy", "flags.npy", "obs.npy", "reward.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES_MAX
    rows = np.load(tmp_path / "a" / "env_index.npy")
    assert rows.dtype == np.float64 and 0 < len(rows) < 100 and np.all(np.diff(rows) > 0)
    for k in arrays:
        a, b = np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy")
        assert np.array_equal(a, b) and np.array_equal(a, arrays[k][rows.astype(int)].astype(a.dtype))


@pytest.mark.gpu
def test_gpu_arm_dumps_the_last_timed_step(tmp_path):
    """--dump-outputs: the same arguments give the same inputs, so two runs write identical outputs."""
    import numpy as np
    n = 4096
    for d in ("a", "b"):
        out = subprocess.run([sys.executable, "bench.py", "--steps", "21", "--warmup", "3", "--no-sweep", "--no-cpu-baseline",
                              "--no-extras", "--envs-per-gpu", str(n), "--dump-outputs", str(tmp_path / d)],
                             cwd=ROOT, capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-3000:]
        assert _one_json_line(out.stdout)["steps"] == 21
    shapes = {"obs": (n, 137), "reward": (n,), "flags": (n,)}
    assert sorted(p.name for p in (tmp_path / "a").iterdir()) == sorted(f"{k}.npy" for k in shapes)
    for k, shape in shapes.items():
        a, b = np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy")
        assert a.shape == shape and a.dtype == np.float32 and np.isfinite(a).all()
        assert np.array_equal(a, b), k
    flags = np.load(tmp_path / "a" / "flags.npy")
    assert set(np.unique(flags)) <= {0.0, 1.0, 2.0, 3.0}


@pytest.mark.gpu
def test_gpu_arm_line():
    out = subprocess.run([sys.executable, "bench.py", "--steps", "30", "--warmup", "3", "--no-sweep", "--no-cpu-baseline",
                          "--no-extras", "--envs-per-gpu", "4096"], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    d = _one_json_line(out.stdout)
    assert BASE_KEYS | {"roofline", "clocks", "substeps_per_sec", "timing_floor_ms", "per_step_flushed"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 30 and d["warmup"] == 3
    assert d["gpu_launches"] == 4 and d["fragment_steps"] == 8      # 30 steps = 3 fragments of 8 + one of 6, one launch each
    assert d["scaling"] == "weak" and d["dtype"] == "f32" and d["data"] == "synthetic" and "workload" in d["config"]
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["bytes_per_env_step"] == 761 and r["units_per_launch"] == 4096 * 8 and r["steps_per_launch"] == 8
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 4096 * 24 and e["d2h_bytes_per_step"] == 4096 * (404 + 4 + 1) and e["value"] > 0
    assert e["sync_full_rows"]["d2h_bytes_per_step"] == 4096 * (548 + 4 + 1) and e["sync_full_rows"]["value"] > 0
    assert abs(d["value"] - 4096 * 30 / (d["ms_per_step"] * 30 / 1e3)) / d["value"] < 1e-6
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert d["episode_stats"]["episodes_total"] > 0            # pre-aged envs: auto-resets happen inside the timed region


@pytest.mark.gpu
def test_gpu_arm_extras_at_a_small_size():
    """The dynamic-mode, obstacle and rollout-loop records are emitted at every world size (here: 1, tiny step count)."""
    out = subprocess.run([sys.executable, "bench.py", "--steps", "16", "--warmup", "3", "--no-sweep", "--no-cpu-baseline",
                          "--envs-per-gpu", "8192"], cwd=ROOT, capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0, out.stderr[-3000:]
    d = _one_json_line(out.stdout)
    assert d["dynamic_mode"]["value"] > 0 and d["dynamic_mode"]["roofline"]["bound"] == "fp32"
    assert d["obstacles"]["kinematic"]["value"] > 0 and d["obstacles"]["dynamic"]["value"] > 0
    assert d["rollout"]["value"] > 0 and d["rollout"]["episode_stats"]["env_steps"] > 0
