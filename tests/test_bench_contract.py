"""bench.py prints exactly ONE JSON line on stdout with the keys the driver reads."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"}


def _run(args, timeout=600):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                       timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--steps", "4", "--warmup", "3", "--cpu-sample-envs", "2048"])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["steps"] == 4
    assert d["metric"] == "env_steps_per_sec" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["vs_baseline"] is None and d["data"] == "synthetic"
    staged = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "inversus_rl", "env_wrappers.py"))
    assert d["cpu_baseline"]["kind"] == ("reference" if staged else "port")  # the reference itself when it is staged
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"] and d["c_port"]["kind"] == "port"
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_prints_the_b200_arm_config_at_every_n():
    """Under torchrun rank 0 of the reference arm describes the workload exactly as the B200 arm does at
    that N (the driver compares the two `config` objects key for key)."""
    sys.path.insert(0, ROOT)
    import bench
    env = dict(os.environ, RANK="0", WORLD_SIZE="2", LOCAL_RANK="0")
    argv = ["--gpus", "2", "--steps", "2", "--warmup", "5", "--cpu-sample-envs", "512"]
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"] + argv,
                       capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    old = sys.argv
    try:
        sys.argv = ["bench.py"] + argv
        want = bench.workload_config(bench.parse_args(), 2)
    finally:
        sys.argv = old
    assert d["config"] == want and d["config"]["total_envs"] == 2 * d["config"]["envs_per_gpu"]
    assert d["config"]["preroll_steps"] == 500 + 100 - 5 and d["n_gpus"] == 2


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--steps", "2", "--warmup", "3", "--cpu-sample-envs", "512"], capture_output=True, text=True,
                       timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_b200_arm_line():
    d = _run(["--envs-per-gpu", "16384", "--steps", "6", "--warmup", "3", "--e2e-steps", "2", "--cpu-seconds", "1",
              "--cpu-sample-envs", "2048", "--ppo", "0"])
    assert BASE_KEYS | {"roofline", "clocks", "e2e_variants"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 6 and d["warmup"] == 3 and d["gpu_launches"] == 6
    assert d["scaling"] == "weak" and d["dtype"] == "u32"
    ro = d["roofline"]
    assert ro["bound"] == "hbm" and ro["unit"] == "GB/s" and abs(ro["frac"] - ro["achieved"] / ro["peak"]) < 1e-9
    assert ro["algorithmic_bytes_per_env_step"] == 7395
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["value"] > 0
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 16384 and e["d2h_bytes_per_step"] > 16384 * 256
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert d["config"]["preroll_steps"] == 500 + 100 - 3       # timed steps lie past the first episode timeout
    ev = d["e2e_variants"]["obs_stay_on_device_episode_events"]
    assert ev["value"] > 0 and ev["d2h_bytes_per_step"] < d["e2e_variants"]["obs_stay_on_device"]["d2h_bytes_per_step"]


def test_reference_arm_refuses_dump_outputs(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--dump-outputs", str(tmp_path / "d")], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and not os.path.exists(tmp_path / "d")


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step_and_reproducible(tmp_path):
    """Two runs with the same arguments write identical files: float32/float64 arrays of the sampled
    envs' outputs of the last timed step, P2's view included in selfplay."""
    import numpy as np
    dumps = []
    for k in range(2):
        out = tmp_path / str(k)
        d = _run(["--mode", "selfplay", "--envs-per-gpu", "300000", "--steps", "5", "--warmup", "3", "--e2e-steps", "0",
                  "--cpu-seconds", "0", "--ppo", "0", "--dump-outputs", str(out)])
        assert d["steps"] == 5 and d["gpu_launches"] == 5
        assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= 64 << 20
        dumps.append({f[:-4]: np.load(out / f) for f in os.listdir(out)})
    a, b = dumps
    assert set(a) == {"env_index", "obs_env_index", "obs", "extra", "reward", "done", "info", "episode_steps",
                      "episode_return", "obs_p2", "extra_p2"}
    assert set(b) == set(a) and all(np.array_equal(a[k], b[k]) for k in a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    rows = a["env_index"]
    assert len(rows) == 1 << 18 and np.all(np.diff(rows) > 0) and rows[-1] < 300000
    assert a["obs"].shape == a["obs_p2"].shape == (2048, 12, 10, 15) and np.isin(a["obs_env_index"], rows).all()
    assert a["reward"].shape == a["done"].shape == (1 << 18,) and a["extra_p2"].shape == (1 << 18, 4)
    assert set(np.unique(a["obs"])) <= {0.0, 1.0} and set(np.unique(a["done"])) <= {0.0, 1.0}


@pytest.mark.gpu
def test_b200_arm_ppo_block():
    """The PPO block of the line (BASELINE.json configs[3] / configs[4] + the labelled epochs=1 run), at toy sizes."""
    d = _run(["--envs-per-gpu", "16384", "--steps", "4", "--warmup", "3", "--e2e-steps", "0", "--cpu-seconds", "0",
              "--ppo", "1", "--ppo-envs3", "2048", "--ppo-envs4", "4096", "--ppo-samples", "32768", "--ppo-iters", "2"],
             timeout=900)
    p = d["ppo"]
    assert p["metric"] == "ppo_samples_per_sec" and p["bf16_peak_tflops"] > 0
    runs = p["runs"]
    assert [r["epochs"] for r in runs] == [4, 4, 1] and [r["mode"] for r in runs] == ["selfplay", "vs_dummy", "vs_dummy"]
    assert "NOT the reference schedule" in runs[2]["run"]
    for r in runs:
        assert r["samples_per_s"] > 0 and r["rollout_env_steps_per_s"] > 0 and r["update_samples_per_s"] > 0
        assert r["iterations_timed"] >= 1 and r["packed_encoder"] is True and r["precision"] == "bf16"
        assert 0 < r["update_frac_of_bf16_sustained"] < 1 and 0 < r["inference_frac_of_bf16_sustained"] < 1
        assert r["allreduce"] is None  # one GPU: no collective
