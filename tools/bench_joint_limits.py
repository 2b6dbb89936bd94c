"""Cost of the joint-limit rows (snk_set_joint_limits) in both kernels with Bullet-order motor rows: the PGS kernel (motor_solver = 0)
and Bullet's literal tick (snk_set_bullet_tick), each with the limits off, on at 1.57 rad (inert on the task's targets) and on at 0.3 rad
(active: the default scaling reaches pi/6), timed alternately in one process with CUDA events; then config 1 (the gait script's raw
ticks, 4 N.m motors) at amplitude 2.2 with the limits off and on at 1.57.  Prints the card and its power limit, then one JSON line.

    python tools/bench_joint_limits.py [--envs 32768] [--steps 3] [--rounds 3] [--gait-replicas 4096] [--gait-ticks 1000]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from bullet_envs_b200 import SnakeVecEnv, default_params, gait_params  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--envs", type=int, default=32768)       # the size of bench.py's bullet_order leg
ap.add_argument("--steps", type=int, default=3)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--gait-replicas", type=int, default=4096)
ap.add_argument("--gait-ticks", type=int, default=1000)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("needs a CUDA device")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print("card:", card or torch.cuda.get_device_name(0), flush=True)


def make(n, bullet_tick, limit, params):
    env = SnakeVecEnv(num_envs=n, device=0, params=params)
    if bullet_tick:
        env.set_bullet_tick(True, 0.1)
    if limit is not None:
        env.set_joint_limits(True, limit)
    env.reset(as_torch=True)
    return env


n = args.envs
g = torch.Generator(device="cuda").manual_seed(0)
acts = torch.rand((args.steps + 1, n, 8), device="cuda", generator=g) * 2 - 1
legs = {}
for kernel, bt in (("pgs", False), ("bullet_tick", True)):
    for tag, limit in (("off", None), ("on_1.57", 1.57), ("on_0.3", 0.3)):
        legs["%s_%s" % (kernel, tag)] = make(n, bt, limit, default_params(motor_solver=0))
res = {k: [] for k in legs}
for env in legs.values():
    env.step(acts[0])                                    # warm-up: module load, caches filled once
torch.cuda.synchronize()
for r in range(args.rounds):
    for name, env in legs.items():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tk = sw = act = 0
        ms = 0.0
        for t in range(args.steps):
            a.record()
            env.step(acts[t + 1])
            b.record(); torch.cuda.synchronize()
            ms += a.elapsed_time(b)
            c = env.counters()
            tk += c["ticks"]; sw += c["pgs_iterations"]
            if not name.endswith("_off"):
                act += env.joint_limit_stats()[0]
        res[name].append({"env_steps_per_s": n * args.steps / ms * 1e3, "ticks_per_s": tk / ms * 1e3, "sweeps_per_tick": sw / tk,
                          "active_rows_per_tick": act / tk})
out = {"card": card, "envs": n, "steps": args.steps, "rounds": args.rounds}
for name, rs in res.items():
    out[name] = {k: [round(x[k], 0 if k.endswith("per_s") else 3) for x in rs] for k in rs[0]}
for env in legs.values():
    env.close()

# config 1: the gait script's open-loop targets at amplitude 2.2 (beyond the +-1.57 limits), raw ticks, every replica the same snake
T, R = args.gait_ticks, args.gait_replicas
nn = np.arange(16)
tg = torch.from_numpy(np.stack([np.where(nn % 2 == 1, -2.2 * np.sin(4 * nn + 2 * k * 0.01), 0.0) for k in range(T)]).astype(np.float32)).cuda()
rows = tg[:, None, :].expand(T, R, 16).contiguous()
for tag, limit in (("off", None), ("on_1.57", 1.57)):
    env = make(R, False, limit, gait_params())
    env.tick(rows[0], 1)                                 # warm-up
    env.reset(hard=True)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    act = tk = 0
    ms = 0.0
    for k in range(T):
        a.record()
        env.tick(rows[k], 1)
        b.record(); torch.cuda.synchronize()
        ms += a.elapsed_time(b)
        tk += R
        if limit is not None:
            act += env.joint_limit_stats()[0]
    s = env.get_state().cpu().numpy()
    out["config1_gait_amp2.2_limits_" + tag] = {"replicas": R, "ticks": T, "env_ticks_per_s": round(R * T / ms * 1e3),
                                                "active_rows_per_tick": round(act / tk, 3), "max_abs_q": round(float(np.abs(s[:, 13:29]).max()), 4),
                                                "replicas_bit_identical": bool((s == s[0]).all())}
    env.close()
print(json.dumps(out))
