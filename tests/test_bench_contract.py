"""bench.py contract on the CPU: the reference arm (the unmodified reference from baseline/_ref on the
host cores; the oracle port when it is not installed) prints exactly one JSON line with the keys a consumer reads.  The
B200 arm needs a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--envs", "64", "--steps", "2",
                          "--warmup", "1", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env-steps/s" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    from oracle.ref_harness import reference_root
    assert d["cpu_baseline"]["kind"] == ("reference" if reference_root() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"]["workload"] == bench.workload_name(64), "both arms must name the workload identically"
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None
    assert d["gae"]["value"] > 0 and d["ppo"]["value"] > 0
    assert list(d)[-2:] == ["ppo", "e2e"], "PPO samples/s and e2e close the line"
    for name, shape in (("obs", (64, 615)), ("privileged_obs", (64, 1050)), ("rewards", (64,)), ("resets", (64,))):
        a = np.load(tmp_path / f"{name}.npy")
        assert a.dtype == np.float32 and a.shape == shape, name


def test_dump_outputs_samples_env_rows_above_64_mib(tmp_path):
    """Outputs above the limit keep a fixed set of env rows, the same rows in every per-env array."""
    sys.path.insert(0, ROOT)
    import bench
    n = 12000                                   # 12000 x 6672 bytes per env row > 64 MB
    ids = torch.arange(n, dtype=torch.float32)
    out = (ids[:, None].expand(n, 615), ids[:, None].repeat(1, 1050), ids.clone(), ids.long() % 2 == 1,
           {"time_outs": ids.long() % 3 == 0, "episode": {"rew_torques": torch.tensor(-0.5)}})
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), out)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["episode_rew_torques.npy", "obs.npy", "privileged_obs.npy", "resets.npy", "rewards.npy", "time_outs.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64_000_000
    got = {f: np.load(tmp_path / "a" / f) for f in files}
    for f in files:
        assert got[f].dtype == np.float32 and np.array_equal(got[f], np.load(tmp_path / "b" / f)), f
    rows = got["rewards.npy"]
    assert 9000 < rows.size < n and np.all(np.diff(rows) > 0)
    assert np.array_equal(got["obs.npy"], np.repeat(rows[:, None], 615, 1))
    assert np.array_equal(got["privileged_obs.npy"][:, -1], rows)
    assert np.array_equal(got["resets.npy"], rows % 2) and np.array_equal(got["time_outs.npy"], (rows % 3 == 0))
    assert got["episode_rew_torques.npy"] == np.float32(-0.5)


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--envs", "64",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
