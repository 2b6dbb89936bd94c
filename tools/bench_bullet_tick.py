"""Bullet's literal tick (snk_set_bullet_tick: Bullet-order motor rows + persistent manifolds + warm start) against the Bullet-order
kernel with the default one-point contacts (motor_solver = 0), timed alternately in one process; then config 1 (the gait script's raw
ticks, 4 N.m motors) with Bullet's contacts.  Prints the card and its power limit, then one JSON line.

    python tools/bench_bullet_tick.py [--envs 32768] [--steps 3] [--rounds 3] [--gait-replicas 4096] [--gait-ticks 1000]
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

n = args.envs
g = torch.Generator(device="cuda").manual_seed(0)
acts = torch.rand((args.steps + 1, n, 8), device="cuda", generator=g) * 2 - 1
legs = {}
bt = SnakeVecEnv(num_envs=n, device=0)
bt.set_bullet_tick(True, 0.1)
legs["bullet_tick"] = bt
legs["bullet_order"] = SnakeVecEnv(num_envs=n, device=0, params=default_params(motor_solver=0))
res = {k: [] for k in legs}
for env in legs.values():
    env.reset(as_torch=True)
    env.step(acts[0])                                    # warm-up: module load, caches filled once
torch.cuda.synchronize()
for r in range(args.rounds):
    for name, env in legs.items():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tk = sw = pts = 0
        ms = 0.0
        for t in range(args.steps):
            a.record()
            env.step(acts[t + 1])
            b.record(); torch.cuda.synchronize()
            ms += a.elapsed_time(b)
            c = env.counters()
            tk += c["ticks"]; sw += c["pgs_iterations"]
            if name == "bullet_tick":
                pts += env.manifold_stats()[0]
        res[name].append({"env_steps_per_s": n * args.steps / ms * 1e3, "ticks_per_s": tk / ms * 1e3, "sweeps_per_tick": sw / tk,
                          "points_per_tick": pts / tk if name == "bullet_tick" else 1.0 * 32})
out = {"card": card, "envs": n, "steps": args.steps, "rounds": args.rounds}
for name, rs in res.items():
    out[name] = {k: [round(x[k], 3 if "per_tick" in k else 0) for x in rs] for k in rs[0]}
for env in legs.values():
    env.close()

# config 1: the gait script's open-loop targets, raw ticks, every replica the same snake
p = gait_params()
T, R = args.gait_ticks, args.gait_replicas
nn = np.arange(16)
tg = torch.from_numpy(np.stack([np.where(nn % 2 == 1, -(np.pi / 6) * np.sin(4 * nn + 2 * k * 0.01), 0.0) for k in range(T)]).astype(np.float32)).cuda()
env = SnakeVecEnv(num_envs=R, device=0, params=p)
env.set_bullet_tick(True, 0.1)
env.reset(as_torch=True)
rows = tg[:, None, :].expand(T, R, 16).contiguous()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
pts = 0
for k in range(T):
    env.tick(rows[k], 1)
    pts += env.manifold_stats()[0]
b.record(); torch.cuda.synchronize()
ms = a.elapsed_time(b)
s = env.get_state().cpu().numpy()
out["config1_gait"] = {"replicas": R, "ticks": T, "env_ticks_per_s": round(R * T / ms * 1e3), "points_per_tick": round(pts / (R * T), 2),
                       "replicas_bit_identical": bool((s == s[0]).all()), "final_base_xy": s[0, 0:2].tolist()}
env.close()
print(json.dumps(out))
