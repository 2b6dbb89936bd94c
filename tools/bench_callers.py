#!/usr/bin/env python3
"""Throughput of the two reference callers on top of the batched env (BASELINE.json configs[2] and [3]).

    python tools/bench_callers.py ppo [--envs 65536]                 # PPO rollout collection (ppo/train.py:112-140)
    torchrun ... tools/bench_callers.py ars [--envs-per-gpu 32768]    # ARS perturbation sweep (ars/train.py:74-116,208-219)

The policies are the callers' (stock torch, out of the kernel scope; restated here because /root/reference does
not exist on the GPU box): ActorCritic 56->256->256->{value, tanh mean, sigmoid+1e-3 std} (ppo/model.py:17-45,
init N(0,0.1)/0.1) and the ARS linear policy a = W_i x, W_i = W + v delta_i (ars/train.py:40-41), one W_i per
environment.  Everything stays on the device: actions are sampled there, the env kernel writes straight into the
rollout buffers, and only the ARS return vector crosses GPUs (one all-gather per rollout)."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def ppo(args):
    import torch
    import torch.nn as nn
    from bullet_envs_b200 import SnakeVecEnv

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    # Normal(mu, sigma) validates its arguments with a device->host synchronisation on every construction (torch._is_all_true): with
    # it the CPU stalls behind every env-step and the ~25 small launches of the policy are exposed; switched off (one line in the
    # caller, ppo/model.py:40-45), the launches run ahead of the GPU and the rollout can be captured as a CUDA graph
    fast = args.no_validate or args.graph
    if args.tf32:  # the caller's choice of matmul precision for its policy (PyTorch default is full fp32)
        torch.backends.cuda.matmul.allow_tf32 = True
    torch.distributions.Distribution.set_default_validate_args(not fast)

    class ActorCritic(nn.Module):
        def __init__(self, ni=56, no=8, hs=(256, 256)):
            super().__init__()
            self.critic = nn.Sequential(nn.Linear(ni, hs[0]), nn.ReLU(), nn.Linear(hs[0], hs[1]), nn.ReLU(), nn.Linear(hs[1], 1))
            self.actor = nn.Sequential(nn.Linear(ni, hs[0]), nn.ReLU(), nn.Linear(hs[0], hs[1]), nn.ReLU())
            self.mu = nn.Linear(hs[1], no)
            self.sigma = nn.Sequential(nn.Linear(hs[1], no), nn.Sigmoid())
            for m in self.modules():
                if isinstance(m, nn.Linear):
                    nn.init.normal_(m.weight, mean=0.0, std=0.1); nn.init.constant_(m.bias, 0.1)

        def forward(self, x):
            h = self.actor(x)
            return torch.distributions.Normal(torch.tanh(self.mu(h)), self.sigma(h) + 0.001), self.critic(x)

    net = ActorCritic().to(dev)
    assert sum(p.numel() for p in net.parameters()) == 165137  # SURVEY.md section 4
    n, T = args.envs, 20  # ppo/params.py:10
    env = SnakeVecEnv(num_envs=n, device=0)
    from bullet_envs_b200.rollout import RolloutBuffer
    buf = RolloutBuffer(T, n, device=dev)
    rew, done = buf.rewards, buf.dones

    def rollout():
        with torch.no_grad():
            for t in range(T):
                dist, v = net(buf.obs[t])
                # dist.sample() is torch.normal(mean, std), which checks std >= 0 with another device->host synchronisation;
                # rsample() (mean + std * randn) draws from the same law without one
                a = dist.rsample() if fast else dist.sample()
                buf.actions[t] = a; buf.log_probs[t] = dist.log_prob(a); buf.values[t] = v.squeeze(-1)
                env.step(a, out=buf.out(t))                      # the kernel writes obs[t+1], rewards[t], dones[t] in place
            _, next_value = net(buf.obs[T])
            returns, adv = buf.gae(next_value.squeeze(-1))         # ppo/agent.py:14-22 as one kernel (snk_gae)
            buf.roll()
        return returns

    buf.obs[0] = env.reset(as_torch=True)
    rollout()  # warm-up
    torch.cuda.synchronize()
    mode = "eager"
    run = rollout
    if args.graph:
        # the whole rollout -- 20 x (policy forward + sample + env-step kernel) + GAE -- captured once as a CUDA graph and replayed:
        # the ~25 small launches per step of the eager policy become one graph launch per rollout
        mode = "cuda graph"
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            rollout()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
            rollout()
        run = g.replay
        run(); torch.cuda.synchronize()

    def timed(fn, reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    ms = timed(run, args.rollouts)
    # breakdown (eager): the env-steps alone on the actions of the last rollout, and the policy alone
    def env_only():
        for t in range(T):
            env.step(buf.actions[t], out=buf.out(t))

    def policy_only():
        with torch.no_grad():
            for t in range(T):
                dist, v = net(buf.obs[t]); a = dist.rsample() if fast else dist.sample(); buf.log_probs[t] = dist.log_prob(a); buf.values[t] = v.squeeze(-1)
            _, nv = net(buf.obs[T]); buf.gae(nv.squeeze(-1))

    ms_env = timed(env_only, 2); ms_pol = timed(policy_only, 2)
    env.close()
    return ({"workload": "PPO rollout collection + GAE (snk_gae), ppo/train.py policy in torch, device-resident RolloutBuffer, " + mode + (", no synchronising argument checks in the policy" if fast else "") + (", tf32 matmul" if args.tf32 else ""), "envs": n, "num_steps": T,
                      "rollouts": args.rollouts, "env_steps_per_s": n * T / (ms * 1e-3), "ms_per_rollout": ms,
                      "ms_env_steps_only": ms_env, "env_steps_per_s_env_only": n * T / (ms_env * 1e-3), "ms_policy_and_gae_only": ms_pol,
                      "ratio_to_env_only": ms_env / ms,
                      "mean_reward": float(rew.mean()), "done_rate": float(done.float().mean()), "n_gpus": 1})


def ars(args):
    import torch
    import torch.distributed as dist
    from bullet_envs_b200 import SnakeVecEnv
    from bullet_envs_b200 import dist as sd

    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    n = args.envs_per_gpu          # = 2 x directions on this GPU: +delta and -delta
    ndir = n // 2
    gen = torch.Generator(device=dev).manual_seed(1000 + rank)  # Philox keyed by rank (directions are sharded)
    delta = torch.randn((ndir, 8, 56), device=dev, generator=gen)
    W = torch.zeros((8, 56), device=dev)
    Wenv = torch.cat([W + 0.03 * delta, W - 0.03 * delta])       # ars/train.py:208-219, v = 0.03
    env = SnakeVecEnv(num_envs=n, device=local)
    if args.manifold is not None:  # Bullet's persistent contact manifolds + warm starting (snk_set_manifold)
        env.set_manifold(True, args.manifold)
    T = 50                                                          # ars/train.py:87
    obs = torch.empty((n, 56), device=dev); rew = torch.empty((n,), device=dev); done = torch.empty((n,), dtype=torch.uint8, device=dev)
    cnt = torch.zeros((), device=dev, dtype=torch.float64); mean = torch.zeros(56, device=dev, dtype=torch.float64); m2 = torch.zeros(56, device=dev, dtype=torch.float64)

    def sweep():
        nonlocal cnt, mean, m2
        ret = torch.zeros((n,), device=dev)
        obs.copy_(env.reset(as_torch=True))
        for t in range(T):
            # running normaliser (ars/train.py:152-169), batch form of Welford
            # the reference's exploration noise on the state, U[0,1) per element (ars/train.py:81,90): without it a
            # zero-mean linear policy never leaves the rest pose (all observations equal their running mean)
            x = (obs + torch.rand(obs.shape, device=dev, generator=gen)).double(); b = x.shape[0]
            bm = x.mean(0); bm2 = ((x - bm) ** 2).sum(0)
            tot = cnt + b; d = bm - mean
            mean = mean + d * b / tot; m2 = m2 + bm2 + d * d * cnt * b / tot; cnt = tot
            std = (m2 / cnt.clamp_min(2)).sqrt().clamp_min(1e-2)
            xn = ((x - mean) / std).float()
            a = torch.bmm(Wenv, xn.unsqueeze(-1)).squeeze(-1)      # one 8x56 mat-vec per environment
            env.step(a, out=(obs, rew, done))
            ret += rew
        full = sd.gather_returns(ret, n * world)                    # the only cross-GPU traffic
        stats = sd.merge_welford(cnt.clone(), mean.clone(), m2.clone())
        return full, stats

    def sweep_fused():
        """the same sweep through snk_rollout_linear: one launch per rollout, normaliser frozen for the rollout (as
        the parallel ARS of Mania et al. does) and updated afterwards from the observation trace"""
        nonlocal cnt, mean, m2
        env.reset(as_torch=True)
        noise = torch.rand((T, n, 56), device=dev, generator=gen)
        std = (m2 / cnt.clamp_min(2)).sqrt().clamp_min(1e-2) if float(cnt) > 0 else torch.ones(56, device=dev, dtype=torch.float64)
        ret, trace = env.rollout_linear(Wenv, T, mean=mean.float(), inv_std=(1.0 / std).float(), noise=noise, trace=True)
        x = trace.view(-1, 56).double(); b = x.shape[0]
        bm = x.mean(0); bm2 = ((x - bm) ** 2).sum(0)
        tot = cnt + b; d = bm - mean
        mean = mean + d * b / tot; m2 = m2 + bm2 + d * d * cnt * b / tot; cnt = tot
        full = sd.gather_returns(ret, n * world)
        stats = sd.merge_welford(cnt.clone(), mean.clone(), m2.clone())
        return full, stats

    if args.fused:
        sweep = sweep_fused
    sweep()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.rollouts):
        full, stats = sweep()
    e1.record(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    if rank == 0:
        print(json.dumps({"workload": "ARS perturbation sweep, linear policy per environment, all-gather of returns" +
                          (", fused rollout kernel (snk_rollout_linear)" if args.fused else ", one env.step per step + policy in torch") +
                          (", persistent contact manifolds, warm start %g" % args.manifold if args.manifold is not None else ""), "envs_total": n * world,
                          "directions": ndir * world, "steps_per_rollout": T, "rollouts": args.rollouts, "n_gpus": world,
                          "env_steps_per_s": n * world * T * args.rollouts / (ms * 1e-3), "ms_per_sweep": ms / args.rollouts,
                          "returns_gathered": int(full.numel()), "mean_return": float(full.mean()), "welford_count": float(stats[0]),
                          "ticks_per_env_step": env.counters()["ticks"] / float(n * T) if args.fused else float(env.last_ticks.float().mean())}))
    env.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("workload", choices=["ppo", "ars"])
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--envs-per-gpu", type=int, default=32768)
    ap.add_argument("--rollouts", type=int, default=3)
    ap.add_argument("--fused", action="store_true", help="ars: run every rollout as one snk_rollout_linear launch")
    ap.add_argument("--manifold", type=float, default=None, metavar="WARM",
                    help="ars: persistent contact manifolds with warm-start factor WARM (env.set_manifold(True, WARM))")
    ap.add_argument("--graph", action="store_true", help="ppo: capture the whole rollout as one CUDA graph")
    ap.add_argument("--tf32", action="store_true", help="ppo: TF32 tensor-core matmuls in the policy")
    ap.add_argument("--no-validate", action="store_true", help="ppo: torch.distributions argument validation off (no per-step synchronisation)")
    a = ap.parse_args()
    res = {"ppo": ppo, "ars": ars}[a.workload](a)
    if res is not None:
        print(json.dumps(res))
