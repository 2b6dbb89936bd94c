"""Joint-limit rows on the GPU (snk_set_joint_limits; the limit block of csrc/snake_pgs.cu, pgs_limit_block) in both kernels with
Bullet-order motor rows -- the PGS kernel (motor_solver = 0) and Bullet's literal tick (snk_set_bullet_tick) -- against the oracle's
rows (Oracle.set_joint_limits; tests/bullet_tick_oracle.py for the literal tick), plus the step paths, checkpoints, refusals, switching
and the release of memory.

Every bar against the fp64 oracle is calibrated in the test itself: the oracle's fp32 build runs the same inputs, and a bar is twice
the fp32 build's separation from the fp64 one plus an fp32 floor (the method of tests/test_gpu_bullet_tick.py).  Horizons stay at
<= 100 raw ticks or a few env-steps: over 300 gait ticks the fp32 and fp64 oracles drift apart by up to 9e-2 rad."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from bullet_envs_b200 import SnakeVecEnv, default_params, gait_params
from bullet_tick_oracle import BulletTickOracle as Oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ["pgs", "bullet_tick"]


@pytest.fixture(scope="module")
def torch():
    import torch as t
    if not t.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU fallback)")
    return t


def make_env(kind, n, params=None, limit=None, mode=None):
    """the PGS kernel (motor_solver = 0 unless params say otherwise) or Bullet's literal tick (warm 0.1), limits at +-limit"""
    env = SnakeVecEnv(num_envs=n, device=0, params=params if params is not None else default_params(motor_solver=0), mode=mode)
    if kind == "bullet_tick":
        env.set_bullet_tick(True, 0.1)
    if limit is not None:
        env.set_joint_limits(True, limit)
    env.reset(as_torch=True)
    return env


def make_oracle(kind, n, params, limit, f32):
    o = Oracle(n, params, f32=f32)
    if kind == "bullet_tick":
        o.set_bullet_tick(True, 0.1)
    o.set_joint_limits(True, limit)
    o.reset()
    return o


def actions(steps, n, seed):
    return np.random.default_rng(seed).uniform(-1, 1, (steps, n, 8)).astype(np.float32)


def gait_targets(ticks, amp):
    nn = np.arange(16)
    return np.stack([np.where(nn % 2 == 1, -amp * np.sin(4 * nn + 2 * k * 0.01), 0.0) for k in range(ticks)]).astype(np.float32)


def separation(ref, got):
    """(tick mismatches, done mismatches, joint error where the ticks agree, median base-position error) over a run, ref = fp64"""
    tick_mis = done_mis = 0
    q = pos = 0.0
    for (o0, d0, t0), (o1, d1, t1) in zip(ref, got):
        same = t0 == t1
        tick_mis += int((~same).sum()); done_mis += int((d0.astype(bool) != d1.astype(bool)).sum())
        if same.any():
            q = max(q, float(np.abs(o0[same, :16] - o1[same, :16]).max()))
        pos = max(pos, float(np.median(np.abs(o0[:, 48:51] - o1[:, 48:51]).max(1))))
    return np.array([tick_mis, done_mis, q, pos], float)


# ---- 1. inert rows change nothing ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_inert_limits_are_bit_identical(torch, kind):
    n = 256
    acts = torch.from_numpy(actions(4, n, 21)).cuda()
    a, b = make_env(kind, n), make_env(kind, n, limit=1.57)
    for t in range(4):
        ra, rb = a.step(acts[t]), b.step(acts[t])
        assert all(torch.equal(x, y) for x, y in zip(ra[:3], rb[:3]))
        assert torch.equal(a.last_ticks, b.last_ticks) and a.counters() == b.counters()
        assert b.joint_limit_stats()[0] == 0
    assert torch.equal(a.get_state(), b.get_state())
    if kind == "bullet_tick":
        assert torch.equal(a.get_manifold_cache(), b.get_manifold_cache())
    a.close(); b.close()
    tg = torch.from_numpy(gait_targets(100, np.pi / 6)).cuda()
    a, b = make_env(kind, 64, gait_params()), make_env(kind, 64, gait_params(), limit=1.57)
    for k in range(100):
        x = tg[k][None].expand(64, 16).contiguous()
        a.tick(x, 1); b.tick(x, 1)
        assert b.joint_limit_stats()[0] == 0
    assert torch.equal(a.get_state(), b.get_state()) and a.counters() == b.counters()
    if kind == "bullet_tick":
        assert torch.equal(a.get_manifold_cache(), b.get_manifold_cache())
    a.close(); b.close()


# ---- 2. active rows against the oracle -----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_active_limits_in_env_steps_against_the_oracle(torch, kind):
    """scaling_factor 2.0 drives the targets past +-1.57: limit rows become active in the env-steps"""
    n, steps = 64, 4
    p = default_params(motor_solver=0, scaling_factor=2.0)
    acts = actions(steps, n, 17)
    ref, act = {}, {}
    for f32 in (False, True):
        o = make_oracle(kind, n, p, 1.57, f32)
        out = []
        for a in acts:
            ob, _, d, tk = o.step(a.astype(np.float64), threads=8)
            out.append((ob, d, tk))
        ref[f32], act[f32] = out, o.row_stats()[1]
        o.close()
    env = make_env(kind, n, p, limit=1.57)
    got, act_g = [], 0
    for a in acts:
        ob, _, d, _ = env.step(torch.from_numpy(a).cuda())
        got.append((ob.cpu().numpy(), d.cpu().numpy(), env.last_ticks.cpu().numpy()))
        act_g += env.joint_limit_stats()[0]
    env.close()
    sep, err = separation(ref[False], ref[True]), separation(ref[False], got)
    bar = 2 * sep + np.array([0.02 * n * steps, 2, 1e-5, 1e-4])
    print("\n%s: fp32 oracle vs fp64 %s, GPU vs fp64 %s; active rows fp64 %d fp32 %d GPU %d" % (kind, sep, err, act[False], act[True], act_g))
    assert act[False] > 0
    assert (err <= bar).all(), (err, bar)
    assert abs(act_g - act[False]) <= 2 * abs(act[True] - act[False]) + 0.01 * act[False] + 2


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("amp,limit", [(2.2, 1.57), (np.pi / 6, 0.4)])
def test_active_limits_in_raw_gait_ticks_against_the_oracle(torch, kind, amp, limit):
    """config 1 (gait_params: 4 N.m motors) at N = 1 for 100 raw ticks, with a gait amplitude beyond the limits.  A joint that hits
    its limit is stopped within a tick, so this trajectory is chaotic: the fp64 oracle started 1e-7 rad away (fp32 rounding of the
    joints) ends up to 0.06-0.3 rad away after 100 ticks, and the fp32 build's separation alone varies tenfold between gaits.  The bar
    therefore takes the largest separation of the fp32 build and of four such perturbed fp64 runs."""
    ticks = 100
    tg = gait_targets(ticks, amp)
    traj = {}
    for f32, seed in ((False, None), (True, None), (False, 0), (False, 1), (False, 2), (False, 3)):
        o = make_oracle(kind, 1, gait_params(), limit, f32)
        if seed is not None:
            s = o.get_state()
            s[0, 13:29] += 1e-7 * np.random.default_rng(seed).standard_normal(16)
            o.set_state(s)
        tr = []
        for k in range(ticks):
            o.tick(tg[k][None].astype(np.float64), 1)
            tr.append(o.get_state()[0].copy())
        traj[(f32, seed)] = np.array(tr)
        o.close()
    ref = traj.pop((False, None))
    env = make_env(kind, 1, gait_params(), limit=limit)
    tr, act = [], 0
    for k in range(ticks):
        env.tick(torch.from_numpy(tg[k][None]).cuda(), 1)
        tr.append(env.get_state()[0].cpu().numpy())
        act += env.joint_limit_stats()[0]
    env.close()
    tr = np.array(tr)
    for sl, fl in ((slice(13, 29), 1e-5), (slice(0, 3), 1e-5)):
        sep = max(np.abs(t[:, sl] - ref[:, sl]).max() for t in traj.values())
        err = np.abs(tr[:, sl] - ref[:, sl]).max()
        assert err <= 2 * sep + fl, (sl, err, sep)
    qmax = np.abs(tr[:, 13:29]).max()
    print("\n%s amp %.3f limit %.2f: max |q| GPU %.4f oracle %.4f, active rows %d" % (kind, amp, limit, qmax, np.abs(ref[:, 13:29]).max(), act))
    assert act > 0
    assert qmax <= (1.60 if limit > 1 else 0.45)                      # the oracle: 1.578 / 1.576 (fp64), 0.407 / 0.421 (fp32)


# ---- 3. every step path runs the same rows -------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_traced_step_and_raw_replicas(torch, kind):
    n = 128
    p = default_params(motor_solver=0, scaling_factor=2.0)
    acts = torch.from_numpy(actions(3, n, 3)).cuda()
    a, b = make_env(kind, n, p, limit=1.57), make_env(kind, n, p, limit=1.57, mode="test")
    for t in range(3):
        ra = a.step(acts[t]); sa = a.joint_limit_stats()
        rb = b.step(acts[t]); sb = b.joint_limit_stats()
        assert all(torch.equal(x, y) for x, y in zip(ra[:3], rb[:3])) and torch.equal(a.last_ticks, b.last_ticks)
        assert a.counters() == b.counters() and sa == sb
    assert sa[0] > 0
    a.close(); b.close()
    n = 4096
    env = make_env(kind, n, gait_params(), limit=1.57)
    tg = torch.from_numpy(gait_targets(100, 2.2)).cuda()
    for k in range(100):
        env.tick(tg[k][None].expand(n, 16).contiguous(), 1)
    s = env.get_state().cpu().numpy()
    env.close()
    assert (s == s[0]).all() and np.abs(s[0, 13:29]).max() > 1.5


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [1000, 1 << 18])
def test_host_path_equals_device_path(torch, kind, n):
    """snk_step_host_f64 (from 2^18 environments its chunks are launches at environment offsets) returns what the device path returns,
    bit for bit, active-row count included"""
    p = default_params(motor_solver=0, scaling_factor=2.0)
    steps = 2 if n < (1 << 18) else 1
    acts = np.random.default_rng(11).uniform(-1, 1, (steps, n, 8)).astype(np.float32)
    a, b = make_env(kind, n, p, limit=1.57), make_env(kind, n, p, limit=1.57)
    for t in range(steps):
        oa, ra, da, _ = a.step(acts[t].astype(np.float64))
        ob, rb, db, _ = b.step(torch.from_numpy(acts[t]).cuda())
        assert np.array_equal(oa.astype(np.float32), ob.cpu().numpy())
        assert np.array_equal(ra.astype(np.float32), rb.cpu().numpy())
        assert np.array_equal(np.asarray(da, bool), db.cpu().numpy().astype(bool))
        assert a.joint_limit_stats() == b.joint_limit_stats()
    assert a.joint_limit_stats()[0] > 0
    assert torch.equal(a.get_state(), b.get_state())
    a.close(); b.close()


@pytest.mark.gpu
def test_chunked_host_path_of_the_exact_kernel_is_unchanged(torch):
    """The active-row count has a counter word of its own, so the chunked snk_step_host_f64 still clears every hand-out word of the
    exact kernel between its launches.  An exact-solver handle on the chunked path (SNK_HOST_FLAGS=0) with the two-pool hand-out
    (SNK_EXACT_SPLIT=0; 2^18 environments in chunks of 65 536, 1.7 waves each, where the short pool's head is counter word 6) returns
    what the device path returns, bit for bit.  In a subprocess: the switches are read once per process."""
    import os, subprocess, sys
    code = ("import numpy as np, torch; from bullet_envs_b200 import SnakeVecEnv\n"
            "n = 1 << 18; acts = np.random.default_rng(5).uniform(-1, 1, (3, n, 8)).astype(np.float32)\n"
            "a, b = SnakeVecEnv(num_envs=n, device=0), SnakeVecEnv(num_envs=n, device=0); a.reset(); b.reset(as_torch=True)\n"
            "for t in range(3):\n"
            "    oa, ra, da, _ = a.step(acts[t].astype(np.float64)); ob, rb, db, _ = b.step(torch.from_numpy(acts[t]).cuda())\n"
            "    assert np.array_equal(oa.astype(np.float32), ob.cpu().numpy()) and np.array_equal(ra.astype(np.float32), rb.cpu().numpy())\n"
            "    assert np.array_equal(np.asarray(da, bool), db.cpu().numpy().astype(bool)) and a.counters() == b.counters()\n"
            "assert torch.equal(a.get_state(), b.get_state()); print('OK')")
    env = dict(os.environ, PYTHONPATH=ROOT, SNK_HOST_FLAGS="0", SNK_EXACT_SPLIT="0")
    out = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert out.returncode == 0 and "OK" in out.stdout, out.stderr[-2000:]


# ---- 4. checkpoints ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_checkpoint_round_trip_and_refused_cross_setting_loads(torch, kind):
    n = 128
    p = default_params(motor_solver=0, scaling_factor=2.0)
    acts = torch.from_numpy(actions(6, n, 9)).cuda()
    a = make_env(kind, n, p, limit=1.57)
    for t in range(3):
        a.step(acts[t])
    sd = a.state_dict()
    assert sd["joint_limit_angle"] == pytest.approx(1.57)
    ref = [a.step(acts[t])[0].clone() for t in range(3, 6)]
    b = make_env(kind, n, p, limit=1.57)
    b.load_state_dict(sd)
    assert all(torch.equal(b.step(acts[t])[0], r) for t, r in zip(range(3, 6), ref))
    off, other = make_env(kind, n, p), make_env(kind, n, p, limit=1.0)
    for env, x in ((off, sd), (other, sd), (a, off.state_dict())):
        before = env.get_state().clone()
        with pytest.raises(ValueError, match="joint limits"):
            env.load_state_dict(x)
        assert torch.equal(env.get_state(), before)
    for env in (a, b, off, other):
        env.close()


# ---- 5. refusals, switching, memory --------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusals_and_switching(torch):
    n = 64
    exact = SnakeVecEnv(num_envs=n, device=0)                       # default parameters: the exact motor solver
    with pytest.raises(RuntimeError, match="motor solver"):
        exact.set_joint_limits(True)
    exact.set_bullet_tick(True, 0.1)
    exact.set_joint_limits(True, 1.57)                                # composes with the literal tick
    with pytest.raises(RuntimeError, match="joint limits off first"):
        exact.set_bullet_tick(False)
    exact.set_joint_limits(False)
    with pytest.raises(RuntimeError, match="joint limits are off"):
        exact.joint_limit_stats()
    exact.set_bullet_tick(False)
    exact.close()
    p = default_params(motor_solver=0, scaling_factor=2.0)
    acts = torch.from_numpy(actions(3, n, 5)).cuda()
    for kind in KINDS:
        env = make_env(kind, n, p)
        for bad in (0.0, -1.0, float("nan"), float("inf")):
            with pytest.raises(RuntimeError, match="angle"):
                env.set_joint_limits(True, bad)
        env.set_joint_limits(True, 0.3)
        on = [tuple(x.clone() for x in env.step(acts[t])[:3]) for t in range(3)]
        env.set_joint_limits(False)
        env.reset(hard=True)
        again = [tuple(x.clone() for x in env.step(acts[t])[:3]) for t in range(3)]
        env.close()
        never = make_env(kind, n, p)
        base = [tuple(x.clone() for x in never.step(acts[t])[:3]) for t in range(3)]
        never.close()
        assert all(all(torch.equal(x, y) for x, y in zip(u, v)) for u, v in zip(again, base))
        assert not all(torch.equal(x, y) for x, y in zip(on[-1], base[-1]))


@pytest.mark.gpu
def test_no_memory_left_behind(torch):
    free = []
    for r in range(6):
        env = make_env(KINDS[r % 2], 4096, limit=1.57)
        env.step(torch.zeros((4096, 8), device="cuda"))
        env.close()
        torch.cuda.synchronize()
        free.append(torch.cuda.mem_get_info()[0])
    free = free[2:]                                                                      # the first rounds load the kernels
    assert max(free) - min(free) <= (4 << 20), free


# ---- 6. SASS of the new kernels (no GPU needed) --------------------------------------------------------------------------------
def test_limit_kernels_have_no_spills_and_sweep_with_indexed_shuffles():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    import __graft_entry__ as ge
    ge.build()
    log = open(os.path.join(ROOT, "bullet_envs_b200", "csrc", "build.log")).read()
    names = ("_Z18snk_lim_env_kernelILb0EE", "_Z18snk_lim_env_kernelILb1EE", "_Z21snk_bt_lim_env_kernelILb0EE", "_Z21snk_bt_lim_env_kernelILb1EE")
    for nm in names:
        blk = log[log.index("Compiling entry function '" + nm):]
        blk = blk[:blk.index("Used ")]
        assert "0 bytes spill stores, 0 bytes spill loads" in blk, blk
    txt = subprocess.check_output([exe, "-sass", os.path.join(ROOT, "bullet_envs_b200", "csrc", "libsnake_b200.so")], text=True)
    for nm in names:
        k = [x for x in txt.split("Function : ") if x.startswith(nm)][0]
        assert k.count("SHFL.IDX") >= 24 and k.count("REDUX") >= 1, (nm, k.count("SHFL.IDX"))
