"""Bullet's literal tick on the GPU (snk_set_bullet_tick, csrc/snake_pgs_manifold.cuh): Bullet-order motor rows together with the
persistent manifolds and warm starting, against the oracle's twin (tests/bullet_tick_oracle.py), plus the traced step, the host paths,
checkpoints, masked hard resets, the switch refusals and the release of the caches.

Every bar against the fp64 oracle is calibrated in the test itself: the oracle's fp32 build runs the same inputs, and a bar is twice
the fp32 build's separation from the fp64 one plus an fp32 floor (the method of tests/test_gpu_manifold.py)."""
import numpy as np
import pytest

from bullet_envs_b200 import SnakeVecEnv, default_params, gait_params
from bullet_tick_oracle import BulletTickOracle as Oracle


@pytest.fixture(scope="module")
def torch():
    import torch as t
    if not t.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU fallback)")
    return t


def bt_env(n, warm=0.1, params=None, mode=None):
    env = SnakeVecEnv(num_envs=n, device=0, params=params, mode=mode)
    env.set_bullet_tick(True, warm)
    env.reset(as_torch=True)
    return env


def actions(steps, n, seed):
    return np.random.default_rng(seed).uniform(-1, 1, (steps, n, 8)).astype(np.float32)


def run_oracle(n, acts, warm, f32):
    o = Oracle(n, default_params(), f32=f32)
    o.set_bullet_tick(True, warm)
    o.reset()
    out = [o.step(a.astype(np.float64), threads=8) for a in acts]
    return out, o.row_stats()[0]


def run_gpu(torch, n, acts, warm):
    env = bt_env(n, warm)
    out, pts, tks = [], 0, 0
    for a in acts:
        obs, rew, done, _ = env.step(torch.from_numpy(a).cuda())
        out.append((obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy(), env.last_ticks.cpu().numpy()))
        p, t = env.manifold_stats(); pts += p; tks += t
    env.close()
    return out, pts / tks


def separation(ref, got):
    """(tick mismatches, done mismatches, joint error where the ticks agree, median base-position error, median reward error without
    the -10 / -5 events) over a run, ref = fp64 oracle"""
    tick_mis = done_mis = 0
    q = pos = rw = 0.0
    for (o0, r0, d0, t0), (o1, r1, d1, t1) in zip(ref, got):
        same = t0 == t1
        tick_mis += int((~same).sum()); done_mis += int((d0.astype(bool) != d1.astype(bool)).sum())
        if same.any():
            q = max(q, float(np.abs(o0[same, :16] - o1[same, :16]).max()))
        pos = max(pos, float(np.median(np.abs(o0[:, 48:51] - o1[:, 48:51]).max(1))))
        ok = (r0 > -4) & (r1 > -4)
        rw = max(rw, float(np.median(np.abs(r0[ok] - r1[ok]))))
    return np.array([tick_mis, done_mis, q, pos, rw], float)


@pytest.mark.gpu
@pytest.mark.parametrize("warm", [0.0, 0.1])
def test_against_the_fp64_oracle(torch, warm):
    n, steps = 128, 8
    acts = actions(steps, n, 7)
    ref, pts64 = run_oracle(n, acts, warm, False)
    f32, pts32 = run_oracle(n, acts, warm, True)
    gpu, ptsg = run_gpu(torch, n, acts, warm)
    sep = separation(ref, f32)
    err = separation(ref, gpu)
    floor = np.array([0.02 * n * steps, 2, 1e-5, 1e-4, 1e-4])
    bar = 2 * sep + floor
    print("\nwarm %.1f  fp32 oracle vs fp64: %s  GPU vs fp64: %s  points/tick %.2f %.2f %.2f" % (warm, sep, err, pts64, pts32, ptsg))
    assert (err <= bar).all(), (err, bar)
    assert abs(ptsg - pts64) <= 2 * abs(pts32 - pts64) + 0.5


@pytest.mark.gpu
def test_raw_gait_ticks_config1(torch):
    """config 1 (the gait script: dt 0.01, 4 N.m motors, so Bullet-order rows) with Bullet's contacts, 100 ticks at N = 1 against the
    oracle; 4 096 replicas stay bit-identical to each other"""
    ticks = 100
    nn = np.arange(16)
    tg = np.stack([np.where(nn % 2 == 1, -(np.pi / 6) * np.sin(4 * nn + 2 * k * 0.01), 0.0) for k in range(ticks)]).astype(np.float32)
    traj = {}
    for f32 in (False, True):
        o = Oracle(1, gait_params(), f32=f32); o.set_bullet_tick(True, 0.1); o.reset()
        tr = []
        for k in range(ticks):
            o.tick(tg[k][None].astype(np.float64), 1)
            tr.append(o.get_state()[0].copy())
        traj[f32] = np.array(tr)
    env = bt_env(1, params=gait_params())
    tr = []
    for k in range(ticks):
        env.tick(torch.from_numpy(tg[k][None]).cuda(), 1)
        tr.append(env.get_state()[0].cpu().numpy())
    tr = np.array(tr)
    env.close()
    for sl, fl in ((slice(13, 29), 1e-5), (slice(0, 3), 1e-5)):
        sep = np.abs(traj[True][:, sl] - traj[False][:, sl]).max()
        err = np.abs(tr[:, sl] - traj[False][:, sl]).max()
        assert err <= 2 * sep + fl, (sl, err, sep)
    n = 4096
    env = bt_env(n, params=gait_params())
    tgt = torch.from_numpy(tg).cuda()
    for k in range(ticks):
        env.tick(tgt[k][None].expand(n, 16).contiguous(), 1)
    s = env.get_state().cpu().numpy()
    env.close()
    assert (s == s[0]).all()


@pytest.mark.gpu
def test_traced_step_equals_the_step_and_matches_the_oracle_trace(torch):
    n = 256
    acts = actions(3, n, 3)
    a, b = bt_env(n), bt_env(n, mode="test")
    for t in range(3):
        oa, ra, da, _ = a.step(torch.from_numpy(acts[t]).cuda()); ca, sa = a.counters(), a.manifold_stats()
        ob, rb, db, info = b.step(torch.from_numpy(acts[t]).cuda()); cb, sb = b.counters(), b.manifold_stats()
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db) and torch.equal(a.last_ticks, b.last_ticks)
        assert torch.equal(a.get_manifold_cache(), b.get_manifold_cache())
        assert ca == cb and sa == sb and sa[0] > 0
        if t == 0:
            first = info
            tk0 = b.last_ticks.cpu().numpy()
    a.close(); b.close()
    ref = {}
    for f32 in (False, True):
        o = Oracle(n, default_params(), f32=f32); o.set_bullet_tick(True, 0.1); o.reset()
        ref[f32] = o.step_trace(acts[0].astype(np.float64))
    sep = err = 0.0
    for e in range(n):
        k = min(int(tk0[e]), int(ref[False][3][e]), int(ref[True][3][e]))
        g = np.array(first[e]["internal_observations"][:k])
        if k:
            sep = max(sep, float(np.abs(ref[True][4][e, :k, :16] - ref[False][4][e, :k, :16]).max()))
            err = max(err, float(np.abs(g[:, :16] - ref[False][4][e, :k, :16]).max()))
    assert err <= 2 * sep + 1e-5, (err, sep)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1000, 1 << 18])
def test_host_path_equals_device_path(torch, n):
    """snk_step_host_f64 (the chunked path: from 2^18 environments its launches start at environment offsets) returns what the device
    path returns, bit for bit"""
    acts = np.random.default_rng(11).uniform(-1, 1, (2, n, 8)).astype(np.float32)
    a, b = SnakeVecEnv(num_envs=n, device=0), SnakeVecEnv(num_envs=n, device=0)
    a.set_bullet_tick(True, 0.1); b.set_bullet_tick(True, 0.1)
    a.reset(); b.reset(as_torch=True)
    for t in range(2):
        oa, ra, da, _ = a.step(acts[t].astype(np.float64))
        ob, rb, db, _ = b.step(torch.from_numpy(acts[t]).cuda())
        assert np.array_equal(oa.astype(np.float32), ob.cpu().numpy())
        assert np.array_equal(ra.astype(np.float32), rb.cpu().numpy())
        assert np.array_equal(np.asarray(da, bool), db.cpu().numpy().astype(bool))
    assert torch.equal(a.get_manifold_cache(), b.get_manifold_cache())
    a.close(); b.close()


@pytest.mark.gpu
def test_checkpoint_resume_cross_model_refusals_and_masked_hard_reset(torch):
    n = 256
    acts = torch.from_numpy(actions(6, n, 9)).cuda()
    a = bt_env(n)
    for t in range(3):
        a.step(acts[t])
    sd = a.state_dict()
    assert sd["bullet_tick_warm"] == 0.1 and tuple(sd["manifold_cache"].shape) == (n, 1056)
    ref = [a.step(acts[t])[0].clone() for t in range(3, 6)]
    b = bt_env(n)
    b.load_state_dict(sd)
    assert all(torch.equal(b.step(acts[t])[0], r) for t, r in zip(range(3, 6), ref))
    c = bt_env(n)
    c.set_state(sd["state"])                                                            # the state without its caches
    assert not all(torch.equal(c.step(acts[t])[0], r) for t, r in zip(range(3, 6), ref))
    # cross-model loads are refused in every direction, before anything is touched
    default = SnakeVecEnv(num_envs=n, device=0); default.reset(as_torch=True)
    man = SnakeVecEnv(num_envs=n, device=0); man.set_manifold(True, 0.1); man.reset(as_torch=True)
    other_warm = bt_env(n, warm=0.0)
    sds = {"default": default.state_dict(), "manifold": man.state_dict(), "bullet": sd}
    for env, own in ((default, "default"), (man, "manifold"), (c, "bullet"), (other_warm, None)):
        before = env.get_state().clone()
        for name, x in sds.items():
            if name == own:
                continue
            with pytest.raises(ValueError, match="contact model"):
                env.load_state_dict(x)
            assert torch.equal(env.get_state(), before)
    # a masked hard reset empties only the masked caches; those environments then match a fresh batch
    mask = torch.zeros(n, dtype=torch.bool); mask[::3] = True
    keep = a.get_manifold_cache()
    a.reset(hard=True, mask=mask.numpy())
    cache = a.get_manifold_cache()
    m = mask.cuda()
    assert (cache[m] == 0).all() and torch.equal(cache[~m], keep[~m])
    fresh = bt_env(n)
    oa, _, _, _ = a.step(acts[0]); of, _, _, _ = fresh.step(acts[0])
    assert torch.equal(oa[m], of[m])
    for env in (a, b, c, default, man, other_warm, fresh):
        env.close()


@pytest.mark.gpu
def test_refusals_and_switching(torch):
    n = 64
    acts = torch.from_numpy(actions(3, n, 5)).cuda()

    def run(env):
        env.reset(as_torch=True)
        return [tuple(x.clone() for x in env.step(acts[t])[:3]) for t in range(3)]

    env = SnakeVecEnv(num_envs=n, device=0)
    base = run(env)
    env.set_bullet_tick(True, 0.1)
    with pytest.raises(RuntimeError, match="snk_set_bullet_tick"):
        env.set_manifold(True, 0.1)
    with pytest.raises(RuntimeError, match="snk_set_bullet_tick"):
        env.rollout_linear(torch.zeros((n, 8, 56), device="cuda"), 2)
    bt2 = run(env)
    env.set_bullet_tick(False)
    again = run(env)
    assert all(all(torch.equal(x, y) for x, y in zip(p, q)) for p, q in zip(base, again))
    env.set_manifold(True, 0.1)
    with pytest.raises(RuntimeError, match="snk_set_manifold"):
        env.set_bullet_tick(True, 0.1)
    env.close()
    with pytest.raises(RuntimeError, match="warm_start"):
        SnakeVecEnv(num_envs=n, device=0).set_bullet_tick(True, -1.0)
    e0 = SnakeVecEnv(num_envs=n, device=0, params=default_params(motor_solver=0))
    e0.set_bullet_tick(True, 0.1)
    bt0 = run(e0)
    e0.close()
    assert all(all(torch.equal(x, y) for x, y in zip(p, q)) for p, q in zip(bt2, bt0))   # motor_solver is not consulted
    assert not torch.equal(bt2[-1][0], base[-1][0])


@pytest.mark.gpu
def test_caches_fill_beyond_45_points_at_rest(torch):
    n = 32
    env = bt_env(n, warm=0.0)
    z = torch.zeros((n, 16), device="cuda")
    env.tick(z, 1)
    p, t = env.manifold_stats()
    assert p == 32 * n and t == n                                                        # first tick: one support vertex per cylinder
    env.tick(z, 150)
    p, t = env.manifold_stats()
    assert p / t > 45
    s = env.get_state().cpu().numpy()
    assert np.isfinite(s).all() and np.abs(s[:, 2]).max() < 3e-3
    env.close()


@pytest.mark.gpu
def test_no_memory_left_behind(torch):
    free = []
    for _ in range(5):
        env = SnakeVecEnv(num_envs=4096, device=0)
        env.set_bullet_tick(True, 0.1)
        env.reset(as_torch=True)
        env.step(torch.zeros((4096, 8), device="cuda"))
        env.close()
        torch.cuda.synchronize()
        free.append(torch.cuda.mem_get_info()[0])
    free = free[1:]                                                                      # the first round loads the kernels
    assert max(free) - min(free) <= (4 << 20), free
