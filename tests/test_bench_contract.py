"""bench.py's contract on the CPU: the reference arm's JSON line (keys the driver parses, honest labels), the workload table
against SURVEY.md section 8's sizes and FLOP counts, and the no-GPU behaviour of the own arm."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_workload_table_matches_the_survey():
    B = bench.WORKLOADS["ppo"]
    assert (B["gym_id"], B["envs_per_gpu"], B["T"], B["nm"], B["epochs"]) == ("CartPole-v1", 65536, 128, 4, 4)
    assert bench.mlp_flops_fwd(B) == 17792                       # SURVEY.md 8(d): fp32 FLOP per env-step, CartPole
    C = bench.WORKLOADS["pendulum"]                               # run_ppo.py:44-51 continuous override
    assert (C["T"], C["nm"], C["epochs"], C["lr"], C["ent"], C["continuous"]) == (256, 32, 10, 3e-4, 0.0, True)
    E = bench.WORKLOADS["scale1m"]
    assert E["total_envs"] == 1048576 and E["scaling"] == "strong" and bench.num_envs_for(E, 8) == 1048576
    assert bench.num_envs_for(B, 8) == 8 * 65536 and bench.GAE_SWEEP_T == (128, 256, 512, 1024, 2048)
    p = bench.params("pendulum", 2, 5)
    assert p["num_envs"] == 131072 and p["continuous"] is True and p["num_minibatches"] == 32 and p["total_timesteps"] == 131072 * 256 * 5
    cfg = bench.workload_config("ppo", 4)
    assert cfg["num_envs"] == 262144 and cfg["num_envs_per_gpu"] == 65536 and "BOUNDED SAMPLE" in cfg["reference_arm_note"]


@pytest.mark.parametrize("workload", ["ppo", "pendulum"])
def test_reference_arm_line(workload):
    env = dict(os.environ, AUR_BENCH_CPU_ENVS="8", OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", workload, "--gpus", "1",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "config", "cpu_baseline", "e2e", "sampled", "host"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_s" and d["unit"] == "env-steps/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # honest labels: the config is the workload the metric is quoted on, the sample that actually ran is spelled out
    want = bench.workload_config(workload, 1)
    assert {k: v for k, v in d["config"].items() if k != "reference_arm_note"} == {k: v for k, v in want.items() if k != "reference_arm_note"}
    assert "num_envs=8" in d["config"]["reference_arm_note"]            # (the test shrank the sample through AUR_BENCH_CPU_ENVS)
    assert d["sampled"]["num_envs"] == 8 and "num_envs=8" in d["cpu_baseline"]["sample"]
    assert d["host"]["torch_num_threads"] >= 1 and "path" in d["host"]     # torch.set_num_threads overrides OMP_NUM_THREADS=1
    if workload == "ppo":
        assert [p["num_envs"] for p in d["cpu_points"]] == [4, 8] and all("rollout_env_steps_per_s" in p for p in d["cpu_points"])


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", AUR_BENCH_CPU_ENVS="8")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_own_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_hidden_dim_flag_reaches_config_params_and_flop_count(monkeypatch):
    """`bench.py --hidden_dim 128 | 256` (src/run_ppo.py:36): the width is named in `config`, handed to ppo(params) and used for
    the algorithmic FLOP count of the roofline; 64 stays the default of every BASELINE config."""
    import bench
    w = bench.WORKLOADS["ppo"]
    assert bench.HIDDEN == 64 and bench.workload_config("ppo", 1)["hidden_dim"] == 64
    f64 = bench.mlp_flops_fwd(w)
    monkeypatch.setattr(bench, "HIDDEN", 128)
    assert bench.workload_config("ppo", 1)["hidden_dim"] == 128 and bench.params("ppo", 1, 3)["hidden_dim"] == 128
    o, a = w["obs"], w["act"]
    assert bench.mlp_flops_fwd(w) == 2 * (o * 128 + 128 * 128 + 128 * a) + 2 * (o * 128 + 128 * 128 + 128) > 3 * f64


def test_dump_outputs_writes_float_arrays_and_samples_large_ones(tmp_path, monkeypatch):
    import numpy as np
    import torch
    monkeypatch.setattr(bench, "DUMP_ELEMENTS", 100)
    small, large = torch.arange(12, dtype=torch.int32).reshape(3, 4), torch.arange(1000, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path), {"small": small, "large": large})
    s, l = np.load(tmp_path / "small.npy"), np.load(tmp_path / "large.npy")
    assert s.dtype == np.float32 and np.array_equal(s, small.numpy())
    assert l.dtype == np.float64 and l.shape == (100,) and np.all(np.diff(l) > 0)
    assert np.array_equal(l, bench.seeded_sample(1000, 100).numpy())           # the same fixed sample every run
    assert np.array_equal(bench.seeded_sample(5, 100).numpy(), np.arange(5))


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_path(tmp_path):
    """Two runs with the same arguments start from the same inputs: the dumped parameters and rollout agree."""
    import numpy as np
    runs = []
    for k in range(2):
        out = tmp_path / str(k)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-cpu-baseline",
                            "--no-extras", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
        runs.append({p.stem: np.load(p) for p in out.glob("*.npy")})
    a, b = runs
    assert sorted(a) == ["actions", "advantages", "dones", "log_probs", "next_value", "obs", "params", "returns", "rewards", "stats",
                         "values"]
    assert sum(v.nbytes for v in a.values()) <= 64 << 20 and all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert a["obs"].shape == (128, bench.DUMP_COLUMNS, 4) and a["stats"].shape == (16, 16)
    assert np.isfinite(a["params"]).all() and np.isfinite(a["advantages"]).all()
    np.testing.assert_allclose(a["params"], b["params"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(a["returns"], b["returns"], rtol=1e-4, atol=1e-4)
