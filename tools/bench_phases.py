#!/usr/bin/env python3
"""Share of the env-step kernel's time in each phase of the physics tick, from the phase clocks of a -DSNK_PHASE_CLOCKS build.

    tools/build_variant.sh phase -DSNK_PHASE_CLOCKS
    python tools/bench_phases.py [--lib bullet_envs_b200/csrc/variants/libsnake_b200_phase.so] [--steps 5 --warmup 2]

Runs the workload of bench.py (2^20 environments, the same seeded U[-1,1] actions, soft-reset start) and prints one JSON line:
per phase the clock64() cycles summed over every warp of every timed launch, and its share of the total.  The clocks are read by
lane 0 of each warp around the phases of ex_tick (snake_exact_core.cuh): pass 1 (tip-ward walk), rows + solver prologue, solver,
pass 2 (base-ward walk) + finish.  A warp's cycles include the issue slots its scheduler gives the other warps, so the shares
are shares of warp residency, which is what the kernel's time is made of when every warp is busy.  The clock reads themselves
cost a few instructions per tick; the kernel time printed beside the shares is the variant's, not the default build's."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PHASES = ["pass 1", "rows + prologue", "solver", "pass 2 + finish"]
CLK_WARPS = 4096


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--lib", default=os.path.join(ROOT, "bullet_envs_b200", "csrc", "variants", "libsnake_b200_phase.so"))
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not os.path.exists(args.lib):
        sys.exit("%s is missing: build it with tools/build_variant.sh phase -DSNK_PHASE_CLOCKS" % args.lib)
    os.environ["SNK_B200_LIB"] = os.path.abspath(args.lib)
    sys.path.insert(0, ROOT)
    import ctypes

    import numpy as np
    import torch

    if not torch.cuda.is_available():
        sys.exit("bench_phases.py needs a CUDA device")
    from bullet_envs_b200 import SnakeVecEnv, _abi
    from bullet_envs_b200 import dist as sd

    lib = _abi.load_library()
    if not hasattr(lib, "snk_phase_clocks"):
        sys.exit("%s has no phase clocks: build it with -DSNK_PHASE_CLOCKS" % args.lib)
    lib.snk_phase_clocks.argtypes = [ctypes.c_void_p, ctypes.c_int]
    dev = torch.device("cuda", 0)
    n, W, K = args.envs, args.warmup, args.steps
    env = SnakeVecEnv(num_envs=n, device=0)
    acts = torch.stack([sd.global_uniform(1234, t, 0, n, 8, dev) for t in range(W + K)])
    obs = torch.empty((n, 56), device=dev); rew = torch.empty((n,), device=dev); done = torch.empty((n,), dtype=torch.uint8, device=dev)
    env.reset(as_torch=True)
    for t in range(W):
        env.step(acts[t], out=(obs, rew, done))
    torch.cuda.synchronize()
    assert lib.snk_phase_clocks(None, 1) == 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ticks = 0
    e0.record()
    for t in range(W, W + K):
        env.step(acts[t], out=(obs, rew, done))
        ticks += int(env.last_ticks.sum().item())
    e1.record()
    torch.cuda.synchronize()
    clk = np.zeros((CLK_WARPS, len(PHASES)), dtype=np.uint64)
    assert lib.snk_phase_clocks(ctypes.c_void_p(clk.ctypes.data), 0) == 0
    per = clk.sum(axis=0).astype(np.float64)
    props = torch.cuda.get_device_properties(0)
    line = {"gpu": props.name, "envs": n, "steps": K, "ticks": ticks, "variant_ms_per_step": e0.elapsed_time(e1) / K,
            "cycles": {p: float(c) for p, c in zip(PHASES, per)},
            "share": {p: round(float(c / per.sum()), 4) for p, c in zip(PHASES, per)}}
    print(json.dumps(line))
    env.close()


if __name__ == "__main__":
    main()
