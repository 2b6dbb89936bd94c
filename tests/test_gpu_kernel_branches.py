"""The env-step's rare branches on every step kernel, against the oracle.  Each kernel has its own copy of the env-step's task logic:

  exact               the thread-per-environment kernel of the exact motor solver (csrc/snake_exact.cu, ex_step_end)
  manifold            snk_set_manifold: persistent manifolds in the exact solver's kernels (man_run + ex_step_end, csrc/snake_manifold.cuh)
  pgs                 motor_solver = 0: the warp-per-environment kernel (env_step, csrc/snake_task.cuh)
  pgs_limits          the same with snk_set_joint_limits
  bullet_tick         snk_set_bullet_tick: Bullet's literal tick (bt_env_step, csrc/snake_pgs_manifold.cuh)
  bullet_tick_limits  the same with snk_set_joint_limits

and the two families decide the branches in different code: per thread in ex_step_end, by a warp-wide vote in the warp kernels.
The branches: the non-finite force-reset (which also empties the environment's contact caches), NaN actions, ragged batch sizes with
clipped actions, height terminations with aborted and live lanes side by side, zero-tick steps, gait_selection 0 and 2,
stale_obs_on_reset, pyramid friction and masked soft / hard resets with persistent manifolds.

Every bar against the fp64 oracle is calibrated in the test itself: the oracle's fp32 build and two fp64 runs perturbed by fp32
rounding's size run the same inputs, and a bar is twice their largest separation from the fp64 run plus an fp32 floor (the method of
tests/test_gpu_joint_limits.py).  An integer outcome that the branch itself forces (a done, 0 or 1 tick, a non-finite count) is
compared exactly."""
import numpy as np
import pytest

from bullet_envs_b200 import SnakeVecEnv, default_params
from bullet_tick_oracle import BulletTickOracle as Oracle

pytestmark = pytest.mark.gpu

KINDS = ["exact", "manifold", "pgs", "pgs_limits", "bullet_tick", "bullet_tick_limits"]
CACHED = ["manifold", "bullet_tick", "bullet_tick_limits"]          # the kinds with persistent contact caches
WARM, LIMIT = 0.1, 1.57
RET, LEN = 62, 63                                                     # SNK_S_RET, SNK_S_LEN


@pytest.fixture(scope="module")
def torch():
    import torch as t
    if not t.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU fallback)")
    return t


def params_of(kind, **kw):
    """the default parameters, with the Bullet-order motor rows (motor_solver = 0) for the warp-per-environment kinds"""
    if kind not in ("exact", "manifold"):
        kw.setdefault("motor_solver", 0)
    return default_params(**kw)


def make_env(kind, n, params, mode=None):
    env = SnakeVecEnv(num_envs=n, device=0, params=params, mode=mode)
    if kind == "manifold":
        env.set_manifold(True, WARM)
    if kind.startswith("bullet_tick"):
        env.set_bullet_tick(True, WARM)
    if kind.endswith("_limits"):
        env.set_joint_limits(True, LIMIT)
    env.reset(as_torch=True)
    return env


def make_oracle(kind, n, params, f32):
    o = Oracle(n, params, f32=f32)
    if kind == "manifold":
        o.set_manifold(True, WARM)
    if kind.startswith("bullet_tick"):
        o.set_bullet_tick(True, WARM)
    if kind.endswith("_limits"):
        o.set_joint_limits(True, LIMIT)
    o.reset()
    return o


class Gpu:
    """a handle behind the interface of Ora: numpy in and out, float64 results, the non-finite count of each step"""

    def __init__(self, torch, kind, n, params, mode=None):
        self.t, self.kind, self.env = torch, kind, make_env(kind, n, params, mode)

    def step(self, a):
        obs, rew, done, _ = self.env.step(self.t.from_numpy(np.ascontiguousarray(a, np.float32)).cuda())
        return (obs.cpu().numpy().astype(np.float64), rew.cpu().numpy().astype(np.float64), done.cpu().numpy().astype(bool),
                self.env.last_ticks.cpu().numpy(), self.env.counters()["nonfinite"])

    def get_state(self):
        return self.env.get_state().cpu().numpy().astype(np.float64)

    def set_state(self, s):
        self.env.set_state(np.ascontiguousarray(s, np.float32))

    def cache(self):
        return self.env.get_manifold_cache().cpu().numpy() if self.kind in CACHED else np.zeros((self.env.num_envs, 0), np.float32)

    def close(self):
        self.env.close()


class Ora:
    """the oracle; seed: the fp64 build with every state it starts from or is given perturbed by 1e-7 rad in the joints (fp32 rounding)"""

    def __init__(self, kind, n, params, f32, seed=None):
        self.o = make_oracle(kind, n, params, f32)
        self.rng = None if seed is None else np.random.default_rng(seed)
        if seed is not None:
            self.set_state(self.get_state())

    def step(self, a):
        before = self.o.counters()["nonfinite"]
        ob, r, d, tk = self.o.step(np.asarray(a, np.float32).astype(np.float64), threads=8)
        return ob.astype(np.float64), r.astype(np.float64), d, tk, self.o.counters()["nonfinite"] - before

    def get_state(self):
        return self.o.get_state().astype(np.float64)

    def set_state(self, s):
        s = np.array(s, np.float64)
        if self.rng is not None:
            s[:, 13:29] += 1e-7 * self.rng.standard_normal((s.shape[0], 16))
        self.o.set_state(s)

    def close(self):
        self.o.close()


def rig(torch, kind, n, params):
    """the fp64 oracle, the calibration runs (the fp32 oracle and two perturbed fp64 oracles), the GPU handle.  With the Bullet-order
    PGS the joints and torques after an env-step depend on which redundant contact carries the load, so a perturbation of fp32
    rounding's size moves them by more than the fp32 build alone shows (the method of test_gpu_joint_limits.py's raw ticks)."""
    return [Ora(kind, n, params, False), Ora(kind, n, params, True), Ora(kind, n, params, False, 0), Ora(kind, n, params, False, 1),
            Gpu(torch, kind, n, params)]


def separation(ref, got):
    """(tick mismatches, done mismatches, joint error where ticks and dones agree, median base-position error, median reward error
    without the penalties) over a run of step outputs, ref = fp64"""
    tick_mis = done_mis = 0
    q = pos = rw = 0.0
    for (o0, r0, d0, t0, _), (o1, r1, d1, t1, _) in zip(ref, got):
        same = (t0 == t1) & (d0 == d1)
        tick_mis += int((t0 != t1).sum()); done_mis += int((d0 != d1).sum())
        if same.any():
            q = max(q, float(np.abs(o0[same, :16] - o1[same, :16]).max()))
        pos = max(pos, float(np.median(np.abs(o0[:, 48:51] - o1[:, 48:51]).max(1))))
        ok = (r0 > -4) & (r1 > -4)
        if ok.any():
            rw = max(rw, float(np.median(np.abs(r0[ok] - r1[ok]))))
    return np.array([tick_mis, done_mis, q, pos, rw], float)


def assert_within_bars(name, runs, n):
    """runs: the step outputs of every member of a rig, in its order"""
    ref, gpu = runs[0], runs[-1]
    sep, err = np.max([separation(ref, c) for c in runs[1:-1]], 0), separation(ref, gpu)
    bar = 2 * sep + np.array([0.02 * n * len(ref) + 1, 2, 1e-5, 1e-4, 1e-4])
    print("\n%s: calibration runs vs fp64 %s, GPU vs fp64 %s" % (name, sep, err))
    assert (err <= bar).all(), (name, err, bar)


def actions(steps, n, seed, scale=1.0, dim=8):
    return (np.random.default_rng(seed).uniform(-1, 1, (steps, n, dim)) * scale).astype(np.float32)


def post_reset_obs(o):
    """the observation of the reset pose (joint slots, base position zero, orientation the identity)"""
    return (o[..., :32] == 0).all(-1) & (o[..., 48:54] == 0).all(-1) & (o[..., 54] == 1)


# ---- 1. a non-finite state is force-reset, and the environment recovers ---------------------------------------------------------
BAD = 7


def nonfinite_run(r, acts, inject=True):
    """one step, s[BAD, 8] = nan, then the other steps; per step its outputs, then the state and the caches (GPU only)"""
    out = []
    for t, a in enumerate(acts):
        if t == 1 and inject:
            s = r.get_state()
            s[BAD, 8] = np.nan
            r.set_state(s)
        out.append(r.step(a) + ((r.get_state(), r.cache()) if isinstance(r, Gpu) else ()))
    return out


@pytest.mark.parametrize("kind", KINDS)
def test_nonfinite_state_is_reset_and_recovers(torch, kind):
    n = 64
    p = params_of(kind)
    acts = actions(5, n, 3, scale=0.5)
    rs = rig(torch, kind, n, p) + [Gpu(torch, kind, n, p)]
    runs = [nonfinite_run(r, acts) for r in rs[:-1]]
    tw = nonfinite_run(rs[-1], acts, inject=False)                      # the twin: the same inputs without the NaN
    for r in rs:
        r.close()
    for run in runs:
        ob, rew, d, _, bad = run[1][:5]
        assert d[BAD] and rew[BAD] == -5.0 and bad == 1 and post_reset_obs(ob[BAD])
        for ob, rew, d, _, bad in (x[:5] for x in run[2:]):
            assert bad == 0 and not d[BAD] and np.isfinite(ob[BAD]).all() and rew[BAD] > -4
    g = runs[-1]
    assert all(np.isfinite(x[5][BAD]).all() for x in g[2:])
    if kind in CACHED:
        assert (g[1][6][BAD] == 0).all()                                  # emptied with the force-reset
        assert (g[0][6][BAD] != 0).any()
    others = np.arange(n) != BAD
    for x, y in zip(g, tw):                                             # every other environment is untouched, bit for bit
        for u, v in zip(x, y):
            if isinstance(u, np.ndarray) and u.ndim:
                assert np.array_equal(u[others], v[others])
    assert_within_bars("non-finite " + kind, [[x[:5] for x in run] for run in runs], n)


def test_nonfinite_state_in_the_manifold_rollout_and_traced_step(torch):
    """snk_rollout_linear and snk_step_trace (mode='test') run the same force-reset as snk_step: one non-finite count, the caches of
    the environment emptied, the other environments untouched"""
    n, T = 64, 4
    p = params_of("manifold")
    acts = torch.from_numpy(actions(1, n, 4, scale=0.5)[0]).cuda()
    a, b = make_env("manifold", n, p), make_env("manifold", n, p)
    for e in (a, b):
        e.step(acts)
    s = a.get_state()
    s[BAD, 8] = float("nan")
    a.set_state(s)
    W = (torch.randn((n, 8, 56), generator=torch.Generator().manual_seed(5)) * 0.05).cuda()
    ra, rb = a.rollout_linear(W, T), b.rollout_linear(W, T)
    assert a.counters()["nonfinite"] == 1 and b.counters()["nonfinite"] == 0
    others = torch.arange(n, device="cuda") != BAD
    assert torch.equal(ra[others], rb[others])
    sa, sb = a.get_state(), b.get_state()
    assert torch.equal(sa[others], sb[others]) and torch.isfinite(sa[BAD]).all()
    assert torch.equal(a.get_manifold_cache()[others], b.get_manifold_cache()[others])
    assert -6.0 < float(ra[BAD]) < -4.0                                 # one -5, then ordinary rewards
    a.close(); b.close()
    # the traced step: the outputs and caches of the plain step, bit for bit, every environment included
    plain, traced = make_env("manifold", n, p), make_env("manifold", n, p, mode="test")
    acts = actions(4, n, 6, scale=0.5)
    for t in range(4):
        if t == 1:
            for e in (plain, traced):
                s = e.get_state()
                s[BAD, 8] = float("nan")
                e.set_state(s)
        x = plain.step(torch.from_numpy(acts[t]).cuda())
        y = traced.step(torch.from_numpy(acts[t]).cuda())
        assert all(torch.equal(u, v) for u, v in zip(x[:3], y[:3])) and torch.equal(plain.last_ticks, traced.last_ticks)
        assert plain.counters() == traced.counters() and plain.counters()["nonfinite"] == (1 if t == 1 else 0)
        cp, ct = plain.get_manifold_cache(), traced.get_manifold_cache()
        assert torch.equal(cp, ct) and (t != 1 or (ct[BAD] == 0).all())
        assert torch.equal(plain.get_state(), traced.get_state())
    plain.close(); traced.close()


# ---- 2. a NaN action ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
def test_nan_action_runs_no_tick(torch, kind):
    """checkBound's comparisons let a NaN through, so the joint error is NaN and checkFeedback ends the loop before the first tick"""
    n, e = 64, 5
    p = params_of(kind)
    acts = actions(2, n, 8, scale=0.5)
    nan = acts.copy()
    nan[1, e, 2] = np.nan
    a, b = Gpu(torch, kind, n, p), Gpu(torch, kind, n, p)
    a.step(nan[0]); b.step(acts[0])
    s0, c0 = a.get_state(), a.cache()
    x, y = a.step(nan[1]), b.step(acts[1])
    s1, c1 = a.get_state(), a.cache()
    others = np.arange(n) != e
    assert x[3][e] == 0 and y[3][e] > 0 and x[4] == 0
    keep = np.ones(s0.shape[1], bool); keep[[RET, LEN]] = False
    assert np.array_equal(s1[e, keep], s0[e, keep]) and s1[e, LEN] == s0[e, LEN] + 1
    assert np.array_equal(c1[e], c0[e])
    for u, v in zip(x[:4], y[:4]):
        assert np.array_equal(u[others], v[others])
    assert np.array_equal(s1[others], b.get_state()[others]) and np.array_equal(c1[others], b.cache()[others])
    a.close(); b.close()
    o = Ora(kind, n, p, False)
    o.step(nan[0])
    assert o.step(nan[1])[3][e] == 0
    o.close()


# ---- 3. ragged batch sizes and clipped actions ----------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [1, 31, 33])
def test_ragged_sizes_with_clipped_actions(torch, kind, n):
    steps = 3
    p = params_of(kind)
    acts = np.random.default_rng(n).permutation(np.linspace(-3, 3, steps * n * 8)).reshape(steps, n, 8).astype(np.float32)
    rs = rig(torch, kind, n, p)
    runs = [[r.step(a) for a in acts] for r in rs]
    clipped = Gpu(torch, kind, n, p)
    cl = [clipped.step(np.clip(a, -1, 1)) for a in acts]
    assert all(all(np.array_equal(u, v) for u, v in zip(x[:4], y[:4])) for x, y in zip(runs[-1], cl))
    assert np.array_equal(rs[-1].get_state(), clipped.get_state())
    for r in rs + [clipped]:
        r.close()
    assert_within_bars("%s n=%d" % (kind, n), runs, n)


# ---- 4. height terminations, aborted and live lanes in one batch ----------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
def test_height_terminations_in_a_batch(torch, kind):
    """the four environments of tests/test_gpu_branches.py side by side: 0 mod 4 untouched; 1 mod 4 lifted by 0.2 m (the height test
    breaks the loop after the first tick); 2 mod 4 thrown upwards (break in the middle of the loop); 3 mod 4 lifted with the action
    already reached (no tick, done by checkTermination's own height test).  Then one more step: an ordinary done keeps the contact
    caches, as Bullet does, and the next step still agrees with the oracle."""
    n = 64
    p = params_of(kind)
    rng = np.random.default_rng(12)
    a0 = rng.uniform(-1, 1, (n, 8)).astype(np.float32)
    a1 = rng.uniform(-1, 1, (n, 8)).astype(np.float32)
    a2 = rng.uniform(-1, 1, (n, 8)).astype(np.float32)
    cls = np.arange(n) % 4
    a1[cls == 3] = a0[cls == 3]
    rs = rig(torch, kind, n, p)
    ref, gpu = rs[0], rs[-1]
    for r in rs:
        r.step(a0)
    s = ref.get_state().astype(np.float32).astype(np.float64)
    s[cls == 1, 2] += 0.2
    s[cls == 2, 9] += rng.uniform(2.5, 3.5, (cls == 2).sum())
    s[cls == 3, 2] += 0.2
    s = s.astype(np.float32).astype(np.float64)
    for r in rs:
        r.set_state(s)
    c0 = gpu.cache()
    out1 = [r.step(a1) for r in rs]
    c1 = gpu.cache()
    out2 = [r.step(a2) for r in rs]
    for r in rs:
        r.close()
    (oo, orr, od, ot, _), (og, rg, dg, tg, _) = out1[0], out1[-1]
    lifted = cls != 0
    for tk, d in ((ot, od), (tg, dg)):
        assert (tk[cls == 1] == 1).all() and (tk[cls == 3] == 0).all() and ((tk[cls == 2] > 1) & (tk[cls == 2] < 20)).all()
        assert d[lifted].all()
    assert (rg[lifted] < -4).all() and post_reset_obs(og[lifted]).all()
    assert np.abs(rg - orr)[cls == 3].max() < 1e-5                     # no tick ran: the closed-form reward
    assert np.array_equal(c1[cls == 3], c0[cls == 3])                  # a done keeps the caches (zero ticks: nothing updated them)
    assert_within_bars("heights " + kind, [[x, y] for x, y in zip(out1, out2)], n)


# ---- 5. zero-tick step ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
def test_zero_tick_step_has_the_closed_form_reward(torch, kind):
    """repeating an action the joints have already reached: checkFeedback is false at once, no tick runs, and the reward is
    calculateReward of the unchanged state"""
    n = 64
    p = params_of(kind)
    a = actions(1, n, 9, scale=0.3)[0]
    g = Gpu(torch, kind, n, p)
    _, _, d0, _, _ = g.step(a)
    s0 = g.get_state()
    target = np.zeros((n, 16))
    target[:, 1::2] = a.astype(np.float64) * p.scaling_factor                # gaitSelection 1: the odd joints
    err = np.sqrt(((target - s0[:, 13:29]) ** 2).sum(1))
    reached = ~d0 & (err < p.err_threshold * (1 - 1e-4))                 # the loop ended on checkFeedback, not a float's width from it
    assert reached.mean() > 0.5, reached.mean()
    _, rew, d, tk, _ = g.step(a)
    s1 = g.get_state()
    g.close()
    assert (tk[reached] == 0).all()
    energy = (s0[:, 29:45] * s0[:, 45:61]).sum(1) * p.energy_dt
    closed = p.alpha * 0.0 + np.where(np.abs(s0[:, 61]) > p.collision_force, p.collision_penalty, 0.0) - p.beta * np.abs(s0[:, 1]) \
        - p.gamma * energy
    closed = closed + np.where(d, p.done_penalty, 0.0)
    assert np.abs(rew - closed)[reached].max() <= 1e-6
    live = reached & ~d
    assert np.array_equal(s1[live][:, :RET], s0[live][:, :RET]) and (s1[live, LEN] == s0[live, LEN] + 1).all()


# ---- 6. gait_selection 0 and 2 --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("gait", [0, 2])
def test_gait_selection_0_and_2(torch, kind, gait):
    """createAction: gaitSelection 0 drives the even (pitch) motors from 8 action dims, 2 all 16 from 16"""
    n, steps = 64, 3
    p = params_of(kind, gait_selection=gait)
    ad = 8 if gait == 0 else 16
    acts = actions(steps, n, 30 + gait, scale=0.5 if gait == 0 else 0.4, dim=ad)
    rs = rig(torch, kind, n, p)
    assert rs[-1].env.act_dim == ad
    runs = [[r.step(a) for a in acts] for r in rs]
    for r in rs:
        r.close()
    assert_within_bars("gait %d %s" % (gait, kind), runs, n)
    for o, _, d, _, _ in (run[-1] for run in (runs[0], runs[-1])):
        live = ~d
        if gait == 0:
            assert np.abs(o[live][:, 0:16:2]).max() > 0.05
        else:
            assert np.abs(o[live][:, 0:16:2]).max() > 0.05 and np.abs(o[live][:, 1:16:2]).max() > 0.05
    if gait == 0:                                                        # the undriven joints stay where the oracle keeps them
        und = [max(np.abs(x[0][~x[2]][:, 1:16:2]).max(initial=0.0) for x in run) for run in runs]
        assert und[-1] <= 2 * max(und[:-1]) + 1e-6, und


# ---- 7. stale_obs_on_reset ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("stale", [0, 1])
def test_torque_slots_after_a_done(torch, kind, stale):
    """stale_obs_on_reset = 1 keeps the last tick's torques and Fz in the post-reset observation (quirk Q9), 0 zeroes them"""
    n = 64
    p = params_of(kind, stale_obs_on_reset=stale)
    a = np.zeros((n, 8), np.float32)
    a[:, 0:5] = 1.0                                                      # drives |q9| past 0.5
    rs = rig(torch, kind, n, p)
    outs = [r.step(a) for r in rs]
    for r in rs:
        r.close()
    for o, _, d, _, _ in outs:
        assert d.all() and (o[:, :32] == 0).all()
        if stale:
            assert np.abs(o[:, 32:48]).max() > 0
        else:
            assert (o[:, 32:48] == 0).all() and (o[:, 55] == 0).all()
    (o0, _, _, t0, _), (og, _, _, tg, _) = outs[0], outs[-1]
    if stale:
        scale = np.abs(o0[:, 32:48]).max()
        sep = max(np.abs(o1 - o0)[t1 == t0][:, 32:48].max(initial=0.0) for o1, _, _, t1, _ in outs[1:-1])
        same = tg == t0
        assert same.mean() > 0.9
        assert np.abs(og - o0)[same][:, 32:48].max() <= 2 * sep + 1e-4 * scale
    assert_within_bars("stale %d %s" % (stale, kind), [[x] for x in outs], n)


# ---- 8. pyramid friction --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
def test_pyramid_friction_env_step(torch, kind):
    """cone_friction = 0 (each friction row clamped on its own): one env-step at moderate actions against the oracle with the same
    switch; the cone's result differs"""
    n = 64
    a = actions(1, n, 41, scale=0.3)[0]
    rs = rig(torch, kind, n, params_of(kind, cone_friction=0))
    outs = [r.step(a) for r in rs]
    for r in rs:
        r.close()
    assert_within_bars("pyramid " + kind, [[x] for x in outs], n)
    cone = Gpu(torch, kind, n, params_of(kind))
    oc = cone.step(a)
    cone.close()
    assert np.median(np.abs(oc[0][:, 48:51] - outs[-1][0][:, 48:51]).max(1)) > 1e-6


# ---- 9. masked soft and hard resets with the caches -----------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["manifold", "bullet_tick"])
@pytest.mark.parametrize("hard", [False, True])
def test_masked_resets_and_the_caches(torch, kind, hard):
    """reset(mask) keeps every cache (a soft reset, as Bullet's); reset(mask, hard=True) empties the masked rows only.  The
    observations equal the oracle's reset(mask) of the same state bit for bit (the hard reset's world rebuild zeroes the state first)."""
    n = 64
    p = params_of(kind)
    env = make_env(kind, n, p)
    for a in actions(2, n, 13, scale=0.5):
        env.step(torch.from_numpy(a).cuda())
    mask = np.arange(n) % 3 == 0
    s = env.get_state().cpu().numpy().astype(np.float64)
    c0 = env.get_manifold_cache().cpu().numpy()
    assert (c0[mask] != 0).any()
    obs = env.reset(torch.from_numpy(mask).cuda(), hard=hard).cpu().numpy()
    c1 = env.get_manifold_cache().cpu().numpy()
    env.close()
    if hard:
        s[mask] = 0.0
        s[mask, 6] = 1.0
        assert (c1[mask] == 0).all() and np.array_equal(c1[~mask], c0[~mask])
    else:
        assert np.array_equal(c1, c0)
    o = make_oracle(kind, n, p, False)
    o.set_state(s)
    ref = o.reset(mask)
    o.close()
    assert np.array_equal(obs, ref.astype(np.float32))
    assert post_reset_obs(obs[mask]).all() and (not hard or (obs[mask][:, 32:48] == 0).all())
