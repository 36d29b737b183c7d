"""CPU (-m "not gpu"): the bench.py contract that can be checked without a GPU -- the reference arm prints exactly ONE
JSON line on stdout with the agreed keys, the workload table / algorithmic-bytes formula match SURVEY 8(d), and
--dump-outputs writes the last step's rows within its size budget.  GPU: two runs of the GPU arm with the same
arguments dump identical outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env-steps/sec" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] == 1
    assert d["value"] > 0 and d["gpu_launches"] == 0 and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["config"]["workload"].startswith("cfg2")
    # both arms print the SAME config object (bench.common_config), including the episode phase the steps are taken from
    sys.path.insert(0, ROOT)
    import bench
    cfg, _, _, envs, D, _, desc = bench.build_workload("cfg2")
    pre = bench.preroll_steps(cfg)
    assert pre > max(cfg.window_size, cfg.scaling_window)
    assert d["config"] == bench.common_config(desc, envs, D, 1, pre) and "steady state" in d["config"]["episode_phase"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "3",
                        "--warmup", "1"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_algorithmic_bytes_formula():
    sys.path.insert(0, ROOT)
    import bench
    want = {"cfg2": 3609, "cfg3": 7209, "cfg4": 4129, "cfg5": 14881}   # SURVEY 8(d)
    for name, (envs, W, strat, rew, pairs, R) in bench.WORKLOADS.items():
        assert 4 * (W * 5 + 2 * W + 4) + 4 + 1 + 4 + R == want[name], name


def _load_dump(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_writes_the_last_step_within_budget(tmp_path, monkeypatch):
    import torch
    sys.path.insert(0, ROOT)
    import bench
    N, D, slots, K = 64, 10, 3, 5
    ring = torch.randn(slots, N, D)
    rews = torch.randn(K, N)
    terms = (torch.rand(K, N) > 0.5).to(torch.uint8)
    equity = torch.randn(N, dtype=torch.float64)

    class Env:
        def info(self):
            return {"equity": equity}

    bench.dump_outputs(str(tmp_path / "full"), Env(), ring, rews, terms, K - 1)
    d = _load_dump(tmp_path / "full")
    assert sorted(d) == ["env_index", "equity", "obs", "reward", "terminated"]
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    np.testing.assert_array_equal(d["obs"], ring[(K - 1) % slots].numpy())
    np.testing.assert_array_equal(d["reward"], rews[K - 1].numpy())
    np.testing.assert_array_equal(d["terminated"], terms[K - 1].numpy().astype(np.float32))
    np.testing.assert_array_equal(d["equity"], equity.numpy())
    np.testing.assert_array_equal(d["env_index"], np.arange(N))

    per_env = 4 * D + 4 + 4 + 8 + 8
    monkeypatch.setattr(bench, "DUMP_BUDGET", 20 * per_env)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), Env(), ring, rews, terms, 1)
    a, b = _load_dump(tmp_path / "a"), _load_dump(tmp_path / "b")
    idx = a["env_index"].astype(np.int64)
    assert len(idx) == 20 and np.all(np.diff(idx) > 0) and sum(v.nbytes for v in a.values()) <= 20 * per_env
    np.testing.assert_array_equal(a["obs"], ring[1].numpy()[idx])
    np.testing.assert_array_equal(a["reward"], rews[1].numpy()[idx])
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)


@pytest.mark.gpu
def test_ours_dump_outputs_are_reproducible(tmp_path):
    """Two runs with the same arguments (503 steps: a 500-step batch, then a 3-step remainder batch whose last step is
    the one dumped) time exactly --steps steps and dump bit-identical outputs of the last one."""
    runs = []
    for run in ("a", "b"):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "503", "--warmup", "2",
                            "--no-single-step", "--no-cpu-baseline", "--no-closed-loop", "--no-other-workloads",
                            "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-2000:]
        line = json.loads(p.stdout)
        assert line["steps"] == 503 and line["value"] > 0
        runs.append(_load_dump(tmp_path / run))
    a, b = runs
    N, D = line["config"]["envs_per_gpu"], line["config"]["obs_dim"]
    assert a["obs"].shape == (N, D) and a["reward"].shape == a["terminated"].shape == a["equity"].shape == (N,)
    assert sum(os.path.getsize(os.path.join(tmp_path, "a", f)) for f in os.listdir(tmp_path / "a")) <= 64_000_000
    assert np.all(np.isfinite(a["obs"])) and np.all(a["equity"] > 0)
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
