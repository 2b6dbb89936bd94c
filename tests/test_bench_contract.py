"""bench.py contract: the reference arm (CPU oracle port) prints one JSON line with the keys a consumer of the benchmark
reads (no GPU needed), and --dump-outputs writes what the timed path computed in its last step (GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0"],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "env-steps/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["steps"] == 1 and line["n_gpus"] == 1
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert "workload" in line["config"]
    # same config object and same tick as this repo's arm (the driver compares the two lines)
    sys.path.insert(0, ROOT)
    import bench
    assert line["config"] == bench.workload_config(1 << 20, 1)
    assert "same tick as the GPU arm" in line["cpu_baseline"]["sample"] and line["cpu_baseline"]["value_bullet_order_rows"] > 0
    assert line["cpu_baseline"]["value"] > line["cpu_baseline"]["value_bullet_order_rows"]   # the relaxed-row tick is the slower one


def test_non_zero_ranks_of_the_reference_arm_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"], env=env,
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr and not os.listdir(tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4096, (1 << 17) + 4096])
def test_dump_outputs_are_the_last_timed_step(tmp_path, n):
    """--dump-outputs writes obs / reward / done / ticks of step W + K - 1 (float32) for the environments of a seed-0 sample of
    DUMP_ENVS ids in ascending order (all of them below DUMP_ENVS): the same values as stepping the seeded actions of bench.py through
    SnakeVecEnv here."""
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU fallback)")
    from bullet_envs_b200 import SnakeVecEnv
    from bullet_envs_b200 import dist as sd
    K, W = 4, 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(K), "--warmup", str(W), "--envs", str(n),
                          "--no-config4", "--no-bullet-order", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == K and line["warmup"] == W
    got = {name: np.load(str(tmp_path / (name + ".npy"))) for name in ("obs", "reward", "done", "ticks")}
    assert sorted(os.listdir(tmp_path)) == sorted(name + ".npy" for name in got)
    assert all(a.dtype == np.float32 for a in got.values())
    env = SnakeVecEnv(num_envs=n, device=0)
    env.reset(as_torch=True)
    for t in range(W + K):
        obs, rew, done, _ = env.step(sd.global_uniform(1234, t, 0, n, 8, torch.device("cuda", 0)))
    dump_envs = 1 << 17
    ids = np.arange(n) if n <= dump_envs else np.sort(np.random.default_rng(0).choice(n, dump_envs, replace=False))
    want = {"obs": obs, "reward": rew, "done": done, "ticks": env.last_ticks}
    for name, a in got.items():
        assert len(a) == len(ids) and np.array_equal(a, want[name].float().cpu().numpy()[ids]), name
    assert got["ticks"].max() >= 1 and np.abs(got["reward"]).max() > 0
    env.close()
