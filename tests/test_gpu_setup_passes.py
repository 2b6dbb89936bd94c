"""Pass 2 of the physics tick (the base-ward walk that yields the applied torques) adds the base-acceleration part to the
wrenches pass 1 computed instead of walking the chain back and recomputing them.  Checked against a build of the library
with -DSNK_PASS2_RECOMPUTE (the recomputing pass 2): 65 536 environments, 20 env-steps from reset, the same seeded actions.
The dynamics do not depend on pass 2, so joints, base, Fz, done and ticks must be bit-identical; the torques and, through the
energy term, the reward may differ at fp32 round-off."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

N, STEPS = 65536, 20

RUNNER = r"""
import hashlib, sys
import numpy as np, torch
sys.path.insert(0, sys.argv[1])
from bullet_envs_b200 import SnakeVecEnv
from bullet_envs_b200 import dist as sd
n, steps = int(sys.argv[3]), int(sys.argv[4])
dev = torch.device("cuda", 0)
env = SnakeVecEnv(num_envs=n, device=0)
obs = torch.empty((n, 56), device=dev); rew = torch.empty((n,), device=dev); done = torch.empty((n,), dtype=torch.uint8, device=dev)
env.reset(as_torch=True)
out = {"same": [], "tau": [], "rew": [], "done": [], "ticks": []}
for t in range(steps):
    env.step(sd.global_uniform(1234, t, 0, n, 8, dev), out=(obs, rew, done))
    o = obs.cpu().numpy()
    out["same"].append(hashlib.sha256(np.ascontiguousarray(np.concatenate([o[:, :32], o[:, 48:]], 1)).tobytes()).hexdigest())
    out["tau"].append(o[:, 32:48]); out["rew"].append(rew.cpu().numpy()); out["done"].append(done.cpu().numpy())
    out["ticks"].append(env.last_ticks.cpu().numpy())
env.close()
np.savez(sys.argv[2], **{k: np.array(v) for k, v in out.items()})
"""


def _run(lib, path):
    env = dict(os.environ, SNK_B200_LIB=lib) if lib else dict(os.environ)
    subprocess.check_call([sys.executable, "-c", RUNNER, ROOT, path, str(N), str(STEPS)], env=env)
    return np.load(path)


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU fallback)")
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge
    ge.build()
    td = tmp_path_factory.mktemp("pass2")
    ref_lib = str(td / "libsnake_b200_recompute.so")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    flags = [f for f in ge.NVCC_FLAGS if f not in ("-Xptxas", "-v")]
    subprocess.check_call([nvcc if os.path.exists(nvcc) else "nvcc"] + flags + ["-DSNK_PASS2_RECOMPUTE", "-o", ref_lib] + ge.SOURCES, cwd=ge.CSRC)
    return _run(None, str(td / "new.npz")), _run(ref_lib, str(td / "ref.npz"))


def test_dynamics_are_bit_identical(runs):
    new, ref = runs
    assert list(new["same"]) == list(ref["same"]), "obs[0:32] / obs[48:56] differ"
    assert np.array_equal(new["done"], ref["done"])
    assert np.array_equal(new["ticks"], ref["ticks"])
    assert new["ticks"].sum() > 0


def test_torques_and_reward_match_at_round_off(runs):
    new, ref = runs
    t_new, t_ref = new["tau"].astype(np.float64), ref["tau"].astype(np.float64)
    assert np.isfinite(t_new).all()
    # relative to the largest torque of the environment and step: a joint that carries almost nothing has no relative precision.
    # The bound is looser than fp32 epsilon because a torque is a small difference of large moments (contact impulses over dt
    # against inertial wrenches), and the two formulations add those in a different order.
    scale = np.abs(t_ref).max(axis=2, keepdims=True)
    rel = np.abs(t_new - t_ref) / np.maximum(scale, 1e-30)
    # reward: absolute for rewards of order one; a reward with the done penalty in it has an fp32 spacing above 1e-5
    r_ref = ref["rew"].astype(np.float64)
    drew = np.abs(new["rew"] - r_ref) / np.maximum(1.0, np.abs(r_ref))
    print("torques: max error relative to the environment's largest torque %.3g (99.9th percentile %.3g); reward: max error %.3g"
          % (rel.max(), np.quantile(rel, 0.999), drew.max()))
    assert rel.max() <= 2e-4, rel.max()
    assert drew.max() <= 1e-5, drew.max()
