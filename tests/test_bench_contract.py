"""bench.py's reference arm runs on the host cores (the CPU restatement of the reference's path): its JSON line can be
checked in the CPU-only container.  The GPU arm is exercised by the driver and by `-m gpu` below."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
        "dtype", "data", "config"}


def run(*args):
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), cwd=ROOT, text=True,
                                  stderr=subprocess.DEVNULL)
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, "bench.py must print exactly one line on stdout"
    return json.loads(lines[0])


def test_reference_arm_json_line():
    d = run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert KEYS <= set(d) and d["impl"] == "reference"
    assert d["unit"] == "env-steps/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["steps"] == 1 and d["warmup"] == 1 and d["vs_baseline"] is None and d["dtype"] == "f64"
    assert "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_uses_every_host_thread_under_torchrun():
    """torchrun exports OMP_NUM_THREADS=1: the round-1 reference arm then ran on ONE core for N > 1."""
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2", LOCAL_RANK="0")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0",
                          "--config", "C2"], capture_output=True, text=True, env=env, timeout=600)
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0)) and d["n_gpus"] == 2
    # ranks other than 0 exit 0 without work and without a line
    env["RANK"] = "1"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_keeps_a_fixed_sample_within_64_mb(tmp_path):
    """--dump-outputs beyond its budget: every array keeps the same seeded sample of environments, in float64, and two
    dumps of the same outputs are identical file for file."""
    import numpy as np
    import bench
    B = 400000
    arrays = {"q": np.random.default_rng(1).normal(size=(B, 7)), "status": np.arange(B, dtype=np.int32),
              "contact_force": np.random.default_rng(2).normal(size=(B, 8, 3))}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted(f.name for f in (tmp_path / "a").iterdir())
    assert files == ["contact_force.npy", "env_index.npy", "q.npy", "status.npy"]
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= 64 * 10**6
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    idx = got["env_index"].astype(np.int64)
    assert 0 < len(idx) < B and (np.diff(idx) > 0).all()
    for name, a in arrays.items():
        assert got[name].dtype == np.float64 and np.array_equal(got[name], a[idx])
    assert all(np.array_equal(np.load(tmp_path / "b" / f), got[f[:-4]]) for f in files)


def test_dump_outputs_below_the_budget_keeps_every_environment(tmp_path):
    import numpy as np
    import bench
    q = np.arange(12.0).reshape(4, 3)
    bench.dump_outputs(str(tmp_path), {"q": q})
    assert np.array_equal(np.load(tmp_path / "q.npy"), q) and np.array_equal(np.load(tmp_path / "env_index.npy"), np.arange(4.0))


@pytest.mark.gpu
def test_gpu_arm_dump_outputs_and_steps(tmp_path):
    """With the same arguments two runs dump identical outputs of their last timed step; --steps sets the number of timed
    steps, in the slow configurations too."""
    import numpy as np
    dumps = []
    for k in range(2):
        d = run("--steps", "12", "--warmup", "3", "--envs", "32768", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / str(k)))
        assert d["steps"] == 12 and d["gpu_launches_detail"]["rkfd_step_kernel"] == 12
        dumps.append({f.name: np.load(f) for f in (tmp_path / str(k)).iterdir()})
    assert set(dumps[0]) == {"q.npy", "qd.npy", "qdd.npy", "status.npy", "contact_active.npy", "contact_type.npy", "contact_ref.npy",
                             "contact_force.npy", "env_index.npy"}
    assert dumps[0]["q.npy"].shape == (32768, 7) and dumps[0]["contact_force.npy"].shape == (32768, 8, 3)
    assert np.isfinite(dumps[0]["q.npy"]).all() and (dumps[0]["status.npy"] == 0).all()
    for name, a in dumps[0].items():
        assert a.dtype == np.float64 and np.array_equal(a, dumps[1][name]), name
    d = run("--steps", "12", "--warmup", "3", "--config", "C4", "--envs", "4096", "--no-cpu-baseline")
    assert d["steps"] == 12 and d["gpu_launches_detail"]["rkfd_step_kernel"] == 12


@pytest.mark.gpu
@pytest.mark.parametrize("config", ["C2", "C5-mlcp", "C5-vert", "C4"])
def test_gpu_arm_other_configs(config):
    d = run("--steps", "3", "--warmup", "3", "--config", config, "--envs", "8192", "--no-cpu-baseline")
    assert d["config"]["name"] == config and d["value"] > 0 and d["gpu_launches_detail"]["rkfd_step_kernel"] == 3
    assert d["gpu_launches"] == 3 + d["gpu_launches_detail"]["resort_kernels"] and ( config != "C4" or d["gpu_launches_detail"]["resorts"] == 3 )
    assert d["roofline_hbm"]["frac"] > 0 and d["e2e"]["value"] > 0


@pytest.mark.gpu
def test_gpu_arm_json_line():
    d = run("--steps", "5", "--warmup", "3", "--envs", "32768")
    assert KEYS <= set(d) and d.get("impl") != "reference"
    assert d["value"] > 0 and d["gpu_launches_detail"]["rkfd_step_kernel"] == 5 and d["steps"] == 5
    assert d["gpu_launches"] == 5 + d["gpu_launches_detail"]["resort_kernels"]
    assert d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    r = d["roofline"]
    # the binding roof of this path is the fp64 pipe (SURVEY.md section 8d); the HBM roofline travels beside it
    assert r["bound"] == "fp64" and 0 < r["frac"] < 1 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    h = d["roofline_hbm"]
    assert h["bound"] == "hbm" and 0 < h["frac"] < 1 and "traffic_note" in h
    assert d["e2e"]["closed_loop_value"] > 0 and d["job_stats"]["envs"] == 32768 and d["job_stats"]["failed_envs"] == 0
    assert d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
