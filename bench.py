#!/usr/bin/env python3
"""bench.py -- snake env-steps/s of the batched SnakeGymEnv.step() hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores
    python bench.py --gpus N --steps K --dump-outputs DIR    # + the outputs of the last timed step as DIR/*.npy

The library is loaded as `python __graft_entry__.py build` left it (a missing or stale one is refused); the benchmark compiles nothing
and writes nothing into the tree.

Workload (BASELINE.json configs[4], SURVEY.md 8d "config 5"): 2^20 environments in total, split
evenly over the N ranks (one process per GPU, no data-path collective -- environments are
independent), fresh U[-1,1]^8 actions every step keyed by (seed, step, global environment index)
and generated on the device before the timed region, soft-reset start.  A "step" is one SubprocVecEnv.step() over the
whole batch = one launch of the fused env-step kernel.

`value`   : env-steps/s with actions and output buffers resident in HBM (CUDA events, max over ranks).
`e2e`     : the same metric through the reference-facing call with HOST buffers -- the default drop-in
            SnakeVecEnv().step(numpy float64) -> C-ABI snk_step_host_f64 (what ppo/train.py:122 calls): actions H2D,
            the kernel, obs/reward/done/ticks D2H, dtype conversion, all inside the timed region.
`roofline`: the env-step kernel against the measured HBM copy bandwidth (MEASURED_PEAKS.json).  The
            kernel keeps an environment on chip for ~30 physics ticks, so its algorithmic bytes are
            tiny by construction (DESIGN.md section 6); `issue` carries the figure that actually
            bounds it (fp32 issue slots).
`cpu_baseline`: the oracle port of the reference algorithm on this box's host cores (rank 0, N=1), same tick as the GPU arm.
`collective` (N>1), `config4_ars_sweep`, `config3_ppo_rollout`, `bullet_order`, `manifold` (N=1): see run_ours.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True  # the tree may be read-only where the benchmark runs: no __pycache__ next to the sources
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TOTAL_ENVS = 1 << 20
WORKLOAD = "1M-env throughput sweep (2^20 envs total, random U[-1,1] actions, 1/240 s ticks, reference defaults)"
SOLVER = "motor rows eliminated (motor_solver=auto -> exact), PGS <= 50 sweeps over 32 contacts, residual 1e-7"
# algorithmic bytes per env-step of the fused kernel (SURVEY.md 8d / DESIGN.md section 6):
# read 45-float minimal state 180 + action 32; write state 180 + obs 224 + reward 4 + done 1
BYTES_PER_ENV_STEP = 621
# fp32 instructions per lane-cycle the CUDA cores can retire: 128 lanes x 2 (FMA) per SM and clock
FP32_FLOP_PER_SM_CLK = 256.0
# environments whose outputs --dump-outputs writes: 2^17 x (56 + 3) float32 = 31 MB
DUMP_ENVS = 1 << 17


def workload_config(total, world):
    """The `config` object of the JSON line: the SAME for this repo's arm and for --impl reference (the driver compares them)."""
    n = total // world
    return {"workload": WORKLOAD, "envs_total": total, "envs_per_gpu": n,
            "actions": "U[-1,1]^8 per env and step, keyed by (seed, step, global env id): identical for any number of ranks",
            "l2": "inputs larger than L2: %.0f MB of state + %.0f MB of outputs per GPU per step vs 126 MB L2" % (n * 256 / 1e6, n * 233 / 1e6),
            "solver": SOLVER}


def ncu_constants():
    """Per-launch counters of the step kernel from the newest committed ncu --set full capture of this command at 2^20 environments
    (profiles/r*_raw_1m.csv; see profiles/README.md): DRAM bytes, warp instructions, issue-active %, FMA-pipe %.  Read at run time so
    that the line never carries numbers of another kernel version; None when no capture is committed."""
    import csv
    import glob
    import re
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r[0-9][0-9]_*raw_1m.csv")),
                   key=lambda f: (int(re.search(r"r(\d+)_", os.path.basename(f)).group(1)), os.path.basename(f)))  # r02_h3 < r02_h4: by name (a checkout does not keep mtimes)
    want = {"dram__bytes_read.sum": "dram_read", "dram__bytes_write.sum": "dram_write", "smsp__inst_executed.sum": "warp_inst",
            "smsp__issue_active.avg.pct_of_peak_sustained_active": "issue_pct", "sm__inst_executed_pipe_fma.avg.pct_of_peak_sustained_active": "fma_pct",
            "smsp__thread_inst_executed_per_inst_executed.ratio": "lanes_per_inst", "launch__registers_per_thread": "regs"}
    for path in reversed(files):
        try:
            rows = list(csv.reader(open(path)))
            hdr = rows[0]
            units = rows[1]
            best = None
            for r in rows[2:]:
                name = r[hdr.index("Kernel Name")]
                if "step_kernel" not in name:
                    continue
                vals = {}
                for col, key in want.items():
                    if col in hdr:
                        v = float(r[hdr.index(col)].replace(",", ""))
                        u = units[hdr.index(col)].lower()
                        v *= {"kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(u, 1.0)
                        vals[key] = v
                if best is None or vals.get("warp_inst", 0) > best.get("warp_inst", 0):
                    best = dict(vals, kernel=name)
            if best and "dram_read" in best:
                best["file"] = os.path.relpath(path, ROOT)
                return best
        except Exception:
            continue
    return None


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.thread.join(timeout=2)
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
                for name, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


def cpu_leg(solver, n_envs, steps, threads, warmup=1):
    """Oracle port on the host cores: `steps` env-steps over n_envs environments after `warmup` steps (the first leaves the rest pose).
    Actions: U[-1,1] per environment and step.  Returns (env-steps/s, ticks/s, seconds)."""
    import numpy as np
    from bullet_envs_b200 import default_params
    from oracle.oracle_py import Oracle
    o = Oracle(n_envs, default_params(motor_solver=solver))
    rng = np.random.default_rng(0)
    o.reset()
    for _ in range(max(1, warmup)):
        o.step(rng.uniform(-1, 1, (n_envs, 8)), threads=threads)
    o.counters(clear=True)
    t0 = time.perf_counter()
    for _ in range(steps):
        o.step(rng.uniform(-1, 1, (n_envs, 8)), threads=threads)
    dt = time.perf_counter() - t0
    c = o.counters()
    o.close()
    return n_envs * steps / dt, c["ticks"] / dt, dt


def run_reference(args):
    """The reference arm: the CPU restatement of the reference algorithm (oracle/snake_oracle.c -- PyBullet itself is not installable in
    this image) on all host cores, with the SAME tick as this repo's arm runs (motor rows eliminated, motor_solver = auto), on a bounded
    sample of the same workload per step.  The Bullet-order variant of the tick (motor rows relaxed inside the PGS) is timed next to
    it on a smaller sample and reported as a second key."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    n = 512 * threads
    v, tk, dt = cpu_leg(2, n, args.steps, threads, warmup=max(1, args.warmup))
    sample = "%d envs x %d env-steps per run (W %d + K %d steps of %d envs), fp64, same tick as the GPU arm (motor rows eliminated), %d host threads" % (
        n, args.steps, args.warmup, args.steps, n, threads)
    nb = 128 * threads
    v0, tk0, dt0 = cpu_leg(0, nb, 2, threads)
    world = max(1, args.gpus)
    line = {"impl": "reference", "metric": "snake env-steps/sec", "value": v, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args.envs, world),
            "ticks_per_s": tk,
            "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": threads, "kind": "port", "sample": sample,
                             "value_bullet_order_rows": v0,
                             "sample_bullet_order_rows": "%d envs x 2 env-steps, fp64, motor rows relaxed inside the PGS in Bullet's order (motor_solver=0; "
                                                         "DESIGN.md D4), %d host threads (%.1f s)" % (nb, threads, dt0)},
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "PyBullet is not installable in this image; this is the C oracle port of the reference algorithm (oracle/snake_oracle.c) "
                    "without the reference's 10 ms sleep per tick (snake.py:296)"}
    print(json.dumps(line))
    return 0


def time_cuda(fn, iters, torch, dist, world, dev):
    """mean milliseconds per call of fn() on the current stream (CUDA events, max over ranks)"""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / iters], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def dump_outputs(path, total, lo, hi, outs, rank, world, dist):
    """--dump-outputs: obs / reward / done / ticks of the last timed step for a fixed sample of DUMP_ENVS global environment ids
    (seed 0, ascending), as float32 `path`/<name>.npy written by rank 0 -- the whole batch would be 2^20 x 59 floats = 247 MB."""
    import numpy as np
    import torch
    ids = np.sort(np.random.default_rng(0).choice(total, min(total, DUMP_ENVS), replace=False))
    rows = torch.as_tensor(ids[(ids >= lo) & (ids < hi)] - lo, device=outs[0].device)
    part = [t[rows].float().cpu().numpy() for t in outs]
    parts = [part]
    if world > 1:
        parts = [None] * world if rank == 0 else None
        dist.gather_object(part, parts, dst=0)  # shards are contiguous and in rank order: the rows stay ascending
    if rank == 0:
        os.makedirs(path, exist_ok=True)
        for i, name in enumerate(("obs", "reward", "done", "ticks")):
            np.save(os.path.join(path, name + ".npy"), np.concatenate([p[i] for p in parts]))


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise RuntimeError("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__ as ge
    from bullet_envs_b200 import SnakeVecEnv, _abi, default_params
    from bullet_envs_b200 import dist as sd
    if _abi.LIB_PATH == ge.LIB and ge._stale(ge.LIB, ge.DEPS):
        raise RuntimeError("%s is missing or older than its sources: run `python __graft_entry__.py build` first "
                           "(the benchmark compiles nothing)" % ge.LIB)

    total = args.envs
    lo, hi = sd.shard_range(total, rank, world)
    n = hi - lo
    K, W = args.steps, args.warmup
    env = SnakeVecEnv(num_envs=n, device=local)
    # actions keyed by (seed, step, GLOBAL environment index): the batch a rank steps does not depend on the number of ranks
    acts = torch.stack([sd.global_uniform(1234, t, lo, hi, 8, dev) for t in range(W + K)])
    obs = torch.empty((n, 56), device=dev); rew = torch.empty((n,), device=dev); done = torch.empty((n,), dtype=torch.uint8, device=dev)
    tick_sum = torch.zeros((), dtype=torch.int64, device=dev)
    env.reset(as_torch=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for t in range(W):
        env.step(acts[t], out=(obs, rew, done))
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = env.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for t in range(W, W + K):
        env.step(acts[t], out=(obs, rew, done))
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    gpu_launches = env.launch_count() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, total, lo, hi, (obs, rew, done, env.last_ticks), rank, world, dist)
    # per-launch kernel time on the launching stream (second pass, one event pair per launch) + tick statistics
    kt = []
    sweeps = 0.0
    for t in range(W, W + K):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); env.step(acts[t], out=(obs, rew, done)); b.record()
        tick_sum += env.last_ticks.sum()
        kt.append((a, b))
    torch.cuda.synchronize()
    kernel_ms = sum(a.elapsed_time(b) for a, b in kt) / len(kt)
    clocks = sampler.stop() if rank == 0 else None
    c = env.counters()
    t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
    stats = torch.tensor([float(tick_sum.item()), float(c["pgs_iterations"]), float(c["ticks"]), float(n)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    ms = float(t_ms.item())
    value = total * K / (ms * 1e-3)
    ticks_per_step_env = stats[0].item() / (K * total)

    # ---- e2e: the reference-facing call with HOST buffers, host<->device traffic inside the timed region every step.
    # Headline = the default drop-in, SnakeVecEnv().step(numpy float64) -> snk_step_host_f64, exactly what ppo/train.py:122 calls.
    Ke = max(1, min(K, args.e2e_steps))
    host_acts = acts[W - 1:W + Ke].cpu().numpy()  # [0] = untimed warm-up action, distinct from the first timed one

    def e2e_leg(e, a_host):
        e.step(a_host[0])  # allocates the staging buffers outside the timed region
        barrier()
        t0 = time.perf_counter()
        for t in range(1, Ke + 1):
            o_h, r_h, d_h, _ = e.step(a_host[t])
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t_e = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
        assert np.isfinite(r_h).all() and o_h.shape == (n, 56)
        return total * Ke / float(t_e.item())

    e2e_value = e2e_leg(env, host_acts.astype(np.float64))
    pinned = SnakeVecEnv(num_envs=n, device=local, obs_dtype=np.float32, pinned_io=True)
    pinned.reset()
    e2e_pinned = e2e_leg(pinned, host_acts)
    pinned.close()

    extra = {}
    # ---- collectives of the callers (SURVEY.md 8e): all-gather of per-environment returns (ars/train.py:113-116) and the Welford
    # all-reduce of the ARS normaliser (ars/train.py:152-169), nccl-tests style: mean microseconds per call, max over ranks
    if world > 1:
        ret = torch.randn((n,), device=dev)
        cnt, mean, m2 = torch.tensor(1000.0 + rank, device=dev, dtype=torch.float64), torch.randn(56, device=dev, dtype=torch.float64), torch.rand(56, device=dev, dtype=torch.float64)
        ag = time_cuda(lambda: sd.gather_returns(ret, total), 50, torch, dist, world, dev)
        out = torch.empty(total, device=dev)
        ag_raw = time_cuda(lambda: dist.all_gather_into_tensor(out, ret), 50, torch, dist, world, dev)
        wf = time_cuda(lambda: sd.merge_welford(cnt, mean, m2), 50, torch, dist, world, dev)
        extra["collective"] = {"backend": "nccl", "ranks": world,
                               "allgather_returns_us": ag * 1e3, "allgather_returns_bytes_per_rank": n * 4,
                               "allgather_returns_call": "dist.gather_returns: size exchange + all_gather_into_tensor of fp32 returns[%d] per rank" % n,
                               "allgather_into_tensor_only_us": ag_raw * 1e3,
                               "welford_allreduce_us": wf * 1e3, "welford_bytes": (1 + 56) * 8 + 56 * 8,
                               "note": "outside the timed region of `value`: the env-step path has no collective (environments are independent)"}

    # ---- config 4 of BASELINE.json: ARS perturbation sweep, 262 144 environments over the ranks, 50-step rollouts fused into one launch
    # per rank (snk_rollout_linear) + NCCL all-gather of the returns.  Directions and state noise keyed by the global environment index.
    if not args.no_config4:
        tot4, T4 = 262144, 50
        lo4, hi4 = sd.shard_range(tot4, rank, world)
        n4 = hi4 - lo4
        ndir = tot4 // 2
        # environment i < ndir runs W + v delta_i, environment ndir + i runs W - v delta_i (ars/train.py:208-219; v = 0.03, W = 0)
        ids = torch.arange(lo4, hi4, device=dev) % ndir
        dlo, dhi = int(ids.min()), int(ids.max()) + 1
        dblock = sd.global_normal(7, 0, dlo, dhi, 8 * 56, dev)
        sign = torch.where(torch.arange(lo4, hi4, device=dev) < ndir, 1.0, -1.0).view(-1, 1)
        Wenv = (0.03 * sign * dblock[ids - dlo]).view(n4, 8, 56).contiguous()
        del dblock
        env4 = SnakeVecEnv(num_envs=n4, device=local)
        noise = torch.stack([(sd.global_uniform(11, t, lo4, hi4, 56, dev) + 1.0) * 0.5 for t in range(T4)])  # U[0,1) state noise, ars/train.py:81,90

        def sweep():
            env4.reset(as_torch=True)
            r = env4.rollout_linear(Wenv, T4, noise=noise)
            return sd.gather_returns(r, tot4)

        full = sweep()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 2
        a.record()
        for _ in range(reps):
            full = sweep()
        b.record(); torch.cuda.synchronize()
        t4 = torch.tensor([a.elapsed_time(b) / reps], dtype=torch.float64, device=dev)
        tk4 = torch.tensor([float(env4.counters()["ticks"])], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t4, op=dist.ReduceOp.MAX)
            dist.all_reduce(tk4, op=dist.ReduceOp.SUM)
        extra["config4_ars_sweep"] = {"envs_total": tot4, "envs_per_gpu": n4, "steps_per_rollout": T4, "ms_per_sweep": float(t4.item()),
                                      "env_steps_per_s": tot4 * T4 / (float(t4.item()) * 1e-3), "ticks_per_env_step": float(tk4.item()) / (tot4 * T4),
                                      "returns_gathered": int(full.numel()), "mean_return": float(full.mean()),
                                      "returns_checksum": float(full.double().sum()),
                                      "call": "snk_rollout_linear (one launch per rank per sweep) + all-gather of returns[%d]" % tot4}
        env4.close()
        del noise, Wenv

    if rank == 0:
        peak, how = _peaks()
        achieved = BYTES_PER_ENV_STEP * n / (kernel_ms * 1e-3) / 1e9
        ncu = ncu_constants()
        variant = _abi.load_library().snk_kernel_variant().decode()
        # the bounds that actually bind: warp-instruction issue slots (4 schedulers x SMs x SM clock) and the fp32 pipe
        sm_hz = ((clocks or {}).get("sm_mhz") or 1965.0) * 1e6
        sms = torch.cuda.get_device_properties(local).multi_processor_count
        tick_rate_per_gpu = (total / world) * ticks_per_step_env / (kernel_ms * 1e-3)
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "peak_source": how, "kernel": variant, "kernel_ms": kernel_ms, "bytes_per_env_step": BYTES_PER_ENV_STEP,
                "note": "not HBM bound by construction: an environment stays on chip (TMEM / shared memory / registers) for ~30 ticks x 32 contacts x <=50 "
                        "solver sweeps per 621 B of HBM traffic; the binding limit is fp32 issue / dependent-issue latency (`issue`, `fp32`; profiles/)"}
        if ncu:
            per_env_tick = ncu["warp_inst"] / (TOTAL_ENVS * 30.03)   # the capture is this command at 2^20 envs, 30.03 ticks per env-step
            bytes_per_env = (ncu["dram_read"] + ncu["dram_write"]) / TOTAL_ENVS
            roof["traffic"] = bytes_per_env * n
            roof["traffic_over_algorithmic"] = bytes_per_env / BYTES_PER_ENV_STEP
            roof["traffic_source"] = "ncu --set full capture %s (kernel %s), per environment x envs per launch here" % (ncu["file"], ncu["kernel"].split("(")[0])
            issue = {"bound": "issue", "achieved": per_env_tick * tick_rate_per_gpu, "peak": 4.0 * sms * sm_hz, "unit": "warp-inst/s",
                     "smsp_issue_active_pct_ncu": ncu.get("issue_pct"), "lanes_per_instruction_ncu": ncu.get("lanes_per_inst"),
                     "source": "warp instructions per env-tick from %s x the tick rate timed here" % ncu["file"]}
            issue["frac"] = issue["achieved"] / issue["peak"]
            roof["issue"] = issue
            fma = ncu.get("fma_pct")
            if fma is not None:
                pk = FP32_FLOP_PER_SM_CLK * sms * sm_hz / 1e12
                roof["fp32"] = {"bound": "fp32 pipe", "fma_pipe_active_pct_ncu": fma, "peak": pk, "unit": "TFLOP/s (all-FMA)", "achieved": fma / 100.0 * pk,
                                "frac": fma / 100.0, "source": ncu["file"]}
        line = {
            "metric": "snake env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(total, world),
            "ticks_per_s": value * ticks_per_step_env, "ticks_per_env_step": ticks_per_step_env,
            "pgs_sweeps_per_tick_last_step": stats[1].item() / max(1.0, stats[2].item()),
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": int(total * 8 * 4),
                    "d2h_bytes_per_step": int(total * (56 * 4 + 4 + 1 + 4)), "steps": Ke,
                    "call": "SnakeVecEnv().step(numpy float64) -> snk_step_host_f64, the default drop-in for ppo/train.py:122: float64 actions in, fresh "
                            "pageable float64 obs / reward arrays out every step (the reference's dtypes); the library narrows the actions into page-locked "
                            "memory, the kernel reads each environment's action row from it and posts obs/reward/done/ticks rows back to page-locked "
                            "memory over PCIe as environments finish, the host threads widen them into the caller's arrays",
                    "value_pinned_f32": e2e_pinned,
                    "call_pinned_f32": "SnakeVecEnv(obs_dtype=float32, pinned_io=True).step(numpy) -> snk_step_host: persistent page-locked result buffers, "
                                       "no dtype conversion (opt-in)"},
            "gpu_launches": int(gpu_launches),
            "roofline": roof,
            "clocks": clocks,
        }
        line.update(extra)
        # The legs below are side measurements next to the headline: a failure of one of them is reported in its key and must not take
        # the line down with it.
        def side_leg(key, fn):
            try:
                line[key] = fn()
            except Exception as ex:  # noqa: BLE001
                line[key] = {"error": "%s: %s" % (type(ex).__name__, ex)}
                try:
                    torch.cuda.synchronize()
                except Exception:  # noqa: BLE001
                    pass

        def leg_hbm():
            # the kernels of the path for which HBM IS the roofline (SURVEY.md 8d): observation epilogue, state copy, GAE scan
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_hbm_kernels
            hb = bench_hbm_kernels.measure(env, iters=20, with_reset=False, peak=peak)
            return {k["kernel"]: {"GB/s": k["GB/s"], "frac": k["frac_of_measured_hbm_peak"], "ms": k["ms"]} for k in hb["kernels"]}

        def leg_bullet_order():
            # the cost of deviation D4 being wrong: the same step with the motor rows relaxed inside the PGS in Bullet's order
            # (motor_solver = 0, warp-per-env kernel), 65 536 environments
            nb = 65536
            eb = SnakeVecEnv(num_envs=nb, device=local, params=default_params(motor_solver=0))
            eb.reset(as_torch=True)
            ab = acts[:3, :nb].contiguous()
            eb.step(ab[0])
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); eb.step(ab[1]); eb.step(ab[2]); b.record(); torch.cuda.synchronize()
            msb = a.elapsed_time(b) / 2
            out = {"envs": nb, "env_steps_per_s": nb / (msb * 1e-3), "ms_per_step": msb, "ticks_per_s": eb.counters()["ticks"] / (msb * 1e-3),
                   "kernel": "snk_env_kernel (warp per environment, 16 motor + 96 contact rows, Bullet's row order, block Gauss-Seidel)",
                   "ratio_to_value": nb / (msb * 1e-3) / value}
            eb.close()
            return out

        def leg_manifold():
            # the cost of deviation D1: the same step with Bullet's persistent contact manifolds and warm starting (snk_set_manifold,
            # csrc/snake_manifold.cuh), 262 144 environments from the reset pose
            nm = 262144
            em = SnakeVecEnv(num_envs=nm, device=local)
            em.set_manifold(True, 0.1)
            em.reset(as_torch=True)
            am = acts[:5, :nm].contiguous()
            em.step(am[0]); em.step(am[1])
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); em.step(am[2]); em.step(am[3]); em.step(am[4]); b.record(); torch.cuda.synchronize()
            msm = a.elapsed_time(b) / 3
            pts, tkm = em.manifold_stats()
            out = {"envs": nm, "env_steps_per_s": nm / (msm * 1e-3), "ms_per_step": msm, "ticks_per_s": tkm / (msm * 1e-3),
                   "contact_points_per_tick": pts / max(tkm, 1), "warm_start": 0.1,
                   "kernel": "snk_man_step_kernel (thread per environment, 4-slot manifold per cylinder, rows in global memory streamed through a "
                             "cp.async ring)",
                   "ratio_to_value": nm / (msm * 1e-3) / value}
            em.close()
            return out

        def leg_config3():
            # config 3 of BASELINE.json: PPO rollout collection, 65 536 environments, the ppo/train.py policy in torch (fp32), 20-step
            # rollouts written in place into the rollout buffer + GAE (snk_gae), captured as one CUDA graph (tools/bench_callers.py)
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import argparse as _ap
            import bench_callers
            r = bench_callers.ppo(_ap.Namespace(envs=65536, rollouts=2, graph=True, tf32=False, no_validate=True))
            return {k: r[k] for k in ("workload", "envs", "num_steps", "env_steps_per_s", "ms_per_rollout", "env_steps_per_s_env_only", "ms_policy_and_gae_only")}

        if world == 1:
            side_leg("hbm_bound_kernels", leg_hbm)
        if world == 1 and not args.no_bullet_order:
            side_leg("bullet_order", leg_bullet_order)
            side_leg("manifold", leg_manifold)
        if world == 1 and not args.no_config4:
            side_leg("config3_ppo_rollout", leg_config3)
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            nb = 2048 * threads  # ~10 s of CPU work per leg
            v2, tk2, dt2 = cpu_leg(2, nb, 2, threads)
            v0, tk0, dt0 = cpu_leg(0, nb // 4, 2, threads)
            line["cpu_baseline"] = {"value": v2, "unit": "env-steps/s", "cores": threads, "kind": "port",
                                    "sample": "oracle fp64, same tick as the GPU arm (motor rows eliminated): %d envs x 2 env-steps (%.1f s)" % (nb, dt2),
                                    "ticks_per_s": tk2, "value_bullet_order_rows": v0,
                                    "sample_bullet_order_rows": "oracle fp64, motor rows relaxed inside the PGS (motor_solver=0): %d envs x 2 env-steps (%.1f s)" % (nb // 4, dt0)}
        print(json.dumps(line))
    env.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=TOTAL_ENVS, help="total environments over all ranks")
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config4", action="store_true")
    ap.add_argument("--no-bullet-order", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write obs / reward / done / ticks of the last timed step (a fixed sample of "
                                                          "%d environments) as DIR/<name>.npy, float32" % DUMP_ENVS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to this repo's arm (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    return run_reference(args) if args.impl == "reference" else run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
