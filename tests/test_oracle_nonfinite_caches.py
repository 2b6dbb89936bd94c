"""The non-finite force-reset with persistent contact manifolds, in the oracle (``Oracle.set_manifold``, and
``BulletTickOracle.set_bullet_tick`` with the joint-limit rows off and on).  An environment whose state goes non-finite is reset and
reported done with the -5 penalty; its contact caches are emptied with it, as a hard reset empties them.  Kept, the caches' non-finite
impulses would warm-start the next solve and the environment would come back non-finite on every later step.  The GPU twins are the
non-finite cells of tests/test_gpu_kernel_branches.py."""
import numpy as np
import pytest

from bullet_envs_b200 import default_params
from bullet_tick_oracle import BulletTickOracle as Oracle

N, BAD, STEPS = 64, 7, 4
KINDS = ["plain", "manifold", "bullet_tick", "bullet_tick_limits"]


def make_oracle(kind):
    o = Oracle(N, default_params(motor_solver=2 if kind in ("plain", "manifold") else 0))
    if kind == "manifold":
        o.set_manifold(True, 0.1)
    if kind.startswith("bullet_tick"):
        o.set_bullet_tick(True, 0.1)
    if kind == "bullet_tick_limits":
        o.set_joint_limits(True, 1.57)
    o.reset()
    return o


def action(t):
    """alternating body waves: the snake stays close to its start pose, so cached points survive the refresh from step to step"""
    a = np.zeros((N, 8))
    a[:, 1] = 0.8 if t % 2 else -0.8
    return a


def run(kind, inject, fresh_from=None):
    """one step, then s[BAD, 8] = nan (inject), then STEPS more; fresh_from = k: a fresh batch fed the actions from step k on"""
    o = make_oracle(kind)
    out = []
    for t in range(STEPS + 1) if fresh_from is None else range(fresh_from, STEPS + 1):
        if t == 1 and inject:
            s = o.get_state()
            s[BAD, 8] = np.nan
            o.set_state(s)
        before = o.counters()["nonfinite"]
        ob, r, d, tk = o.step(action(t), threads=8)
        out.append((ob, r, d, tk, o.counters()["nonfinite"] - before, o.get_state()))
    o.close()
    return out


@pytest.mark.parametrize("kind", KINDS)
def test_a_force_reset_environment_recovers(kind):
    got, twin = run(kind, True), run(kind, False)
    ob, r, d, _, bad, _ = got[1]
    assert d[BAD] and r[BAD] == -5.0 and bad == 1
    assert (ob[BAD, :32] == 0).all() and (ob[BAD, 48:51] == 0).all() and ob[BAD, 54] == 1
    for ob, r, d, tk, bad, s in got[2:]:
        assert bad == 0 and not d[BAD] and r[BAD] > -4 and np.isfinite(s[BAD]).all()
    others = np.arange(N) != BAD
    for g, w in zip(got, twin):                                   # the other environments never see the injection
        for x, y in zip(g[:4] + g[5:], w[:4] + w[5:]):
            assert np.array_equal(x[others], y[others])


@pytest.mark.parametrize("kind", KINDS)
def test_a_force_reset_environment_restarts_like_a_fresh_one(kind):
    """from the step after the force-reset, the environment's outputs and state are those of a freshly created batch fed the same
    actions, bit for bit: the reset pose and, with persistent manifolds, empty caches"""
    got, fresh = run(kind, True), run(kind, False, fresh_from=2)
    for g, f in zip(got[2:], fresh):
        for x, y in zip(g[:4] + g[5:], f[:4] + f[5:]):
            assert np.array_equal(x[BAD], y[BAD])
