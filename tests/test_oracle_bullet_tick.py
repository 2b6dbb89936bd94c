"""Bullet's literal tick in the oracle (``BulletTickOracle.set_bullet_tick``, tests/oracle_bt/bullet_tick_oracle.c on top of the unchanged oracle): the Bullet-order tick (motor rows relaxed in the PGS, deviation
D4 lifted) on the contact set of the persistent manifolds (deviation D1 lifted), normal impulses warm-started.  Test infrastructure:
the CUDA twin is ``snk_set_bullet_tick`` (tests/test_gpu_bullet_tick.py)."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from bullet_envs_b200 import default_params
from bullet_tick_oracle import BulletTickOracle as Oracle
from oracle.oracle_py import Oracle as PlainOracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_steps(o, acts):
    o.reset()
    out = [o.step(a) for a in acts]
    return [np.concatenate([x[0].ravel(), x[1].ravel(), x[2].ravel(), x[3].ravel()]) for x in out], o.get_state()


def acts_of(n, steps, seed=0):
    return np.random.default_rng(seed).uniform(-1, 1, (steps, n, 8))


@pytest.mark.parametrize("solver", [0, 2])
def test_switching_off_restores_the_original_solver_bit_for_bit(solver):
    acts = acts_of(4, 4)
    fresh = PlainOracle(4, default_params(motor_solver=solver))
    ref, sref = run_steps(fresh, acts)
    o = Oracle(4, default_params(motor_solver=solver))
    o.set_bullet_tick(True, 0.1)
    run_steps(o, acts[:2])
    o.set_bullet_tick(False)
    got, sgot = run_steps(o, acts)
    assert all(np.array_equal(a, b) for a, b in zip(ref, got)) and np.array_equal(sref, sgot)


def test_the_switch_composes_on_any_handle_and_ignores_motor_solver():
    acts = acts_of(4, 3, seed=5)
    outs = []
    for solver in (0, 2):
        o = Oracle(4, default_params(motor_solver=solver))
        o.set_bullet_tick(True, 0.1)
        outs.append(run_steps(o, acts))
    assert all(np.array_equal(a, b) for a, b in zip(outs[0][0], outs[1][0])) and np.array_equal(outs[0][1], outs[1][1])
    o = PlainOracle(4, default_params(motor_solver=0))
    plain, _ = run_steps(o, acts)
    assert not all(np.array_equal(a, b) for a, b in zip(plain, outs[0][0]))     # the manifolds change the contact set


def test_warm_start_changes_the_trajectory():
    acts = acts_of(2, 4, seed=2)
    res = []
    for warm in (0.0, 0.1):
        o = Oracle(2, default_params())
        o.set_bullet_tick(True, warm)
        res.append(run_steps(o, acts)[1])
    assert not np.array_equal(res[0], res[1])


def test_each_switch_refuses_while_the_other_is_on():
    o = Oracle(1, default_params())
    o.set_bullet_tick(True, 0.1)
    with pytest.raises(RuntimeError):
        o.set_manifold(True, 0.1)
    o.set_bullet_tick(False)
    o.set_manifold(True, 0.1)
    with pytest.raises(ValueError):
        o.set_bullet_tick(True, 0.1)
    o2 = Oracle(1, default_params())
    with pytest.raises(ValueError):
        o2.set_bullet_tick(True, -0.1)


def test_caches_fill_at_rest_and_break_when_sliding():
    o = Oracle(1, default_params()); o.set_bullet_tick(True, 0.0); o.reset()
    o.tick(np.zeros((1, 16)), 1)
    assert o.row_stats()[0] == 32                                                      # first tick: one support vertex per cylinder
    o.tick(np.zeros((1, 16)), 150)
    assert o.row_stats()[0] > 45
    s = o.get_state()
    assert np.isfinite(s).all() and abs(s[0, 2]) < 3e-3                                # resting on the plane (margin 1 mm)
    o2 = Oracle(1, default_params()); o2.set_bullet_tick(True, 0.0); o2.reset()
    tg = np.zeros((1, 16)); tg[0, 1::2] = 0.5
    o2.tick(tg, 60)
    assert o2.row_stats()[0] < 45                                                      # sliding contacts drift off their anchors


def test_joint_limit_rows_stay_inert_in_the_composed_tick():
    acts = acts_of(8, 4, seed=3)
    outs = []
    for lim in (False, True):
        o = Oracle(8, default_params())
        o.set_bullet_tick(True, 0.1)
        if lim:
            o.set_joint_limits(True)
        outs.append(run_steps(o, acts))
        if lim:
            assert o.row_stats()[1] == 0
    assert all(np.array_equal(a, b) for a, b in zip(outs[0][0], outs[1][0])) and np.array_equal(outs[0][1], outs[1][1])


def test_composed_tick_against_pybullet(capsys):
    """The fourth row next to tests/test_pybullet_live.py::test_which_variant_matches_pybullet: the composed tick is Bullet's own by
    construction.  Runs wherever PyBullet imports."""
    pybullet = pytest.importorskip("pybullet")
    pybullet_data = pytest.importorskip("pybullet_data")
    from bullet_envs_b200.urdf_model import DEFAULT_URDF, build_model
    p = pybullet
    cid = p.connect(p.DIRECT)
    try:
        p.setAdditionalSearchPath(pybullet_data.getDataPath())
        p.resetSimulation()
        p.setGravity(0, 0, -9.8)
        p.setTimeStep(1.0 / 240)
        p.loadURDF("plane.urdf")
        snake = p.loadURDF(DEFAULT_URDF, [0, 0, 0], flags=p.URDF_USE_SELF_COLLISION)
        motors = build_model().motor_joint_indices
        for j in range(p.getNumJoints(snake)):
            p.setJointMotorControl2(snake, j, p.VELOCITY_CONTROL, force=0)
        acts = np.random.default_rng(1).uniform(-1, 1, (10, 8))
        o = Oracle(1, default_params())
        o.set_bullet_tick(True, 0.1)
        o.reset()
        dt, dp = 0, 0.0
        for a in acts:
            tgt = np.zeros(16); tgt[1::2] = a * np.pi / 6
            ticks = 0
            while True:
                q = np.array([p.getJointState(snake, j)[0] for j in motors])
                if not np.linalg.norm(tgt - q) > 0.05 or ticks > 40:
                    break
                p.setJointMotorControlArray(snake, motors, p.POSITION_CONTROL, targetPositions=list(tgt), forces=[np.inf] * 16)
                p.stepSimulation()
                ticks += 1
            pos, _ = p.getBasePositionAndOrientation(snake)
            ob, _, _, ot = o.step(a[None, :])
            dt += abs(int(ot[0]) - ticks)
            dp = max(dp, float(np.abs(ob[0, 48:51] - np.array(pos)).max()))
    finally:
        p.disconnect(cid)
    with capsys.disabled():
        print("\n%-55s %6d %12.4f" % ("Bullet tick (Bullet-order rows, manifolds + warm 0.1)", dt, dp))
    assert dp < 0.1


def test_new_kernels_have_no_spills_and_broadcast_with_indexed_shuffles(tmp_path):
    """SASS of the composed tick's kernels (no GPU needed): 0 spill bytes in ptxas, and the block Gauss-Seidel broadcasts one impulse
    change per row with SHFL.IDX"""
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    import __graft_entry__ as ge
    ge.build()
    log = open(os.path.join(ROOT, "bullet_envs_b200", "csrc", "build.log")).read()
    names = ("snk_bt_env_kernelILb0EE", "snk_bt_env_kernelILb1EE")
    for nm in names:
        blk = log[log.index("Compiling entry function '_Z17" + nm):]
        blk = blk[:blk.index("Used ")]
        assert "0 bytes spill stores, 0 bytes spill loads" in blk, blk
    txt = subprocess.check_output([exe, "-sass", os.path.join(ROOT, "bullet_envs_b200", "csrc", "libsnake_b200.so")], text=True)
    for nm in names:
        k = [p for p in txt.split("Function : ") if p.startswith("_Z17" + nm)][0]
        assert k.count("SHFL.IDX") >= 20 and k.count("REDUX") >= 1, k.count("SHFL.IDX")
