"""Known answer of the oracle's joint-limit rows (Oracle.set_joint_limits, the specification of snk_set_joint_limits): a finite motor
that pushes a yaw joint past a tight limit is held at the limit, saturated, with limit rows active.  CPU only."""
import numpy as np
import pytest

from bullet_envs_b200 import gait_params
from oracle.oracle_py import Oracle


@pytest.mark.parametrize("joint", [1, 5])
@pytest.mark.parametrize("sign", [1.0, -1.0])
def test_a_saturated_motor_is_held_at_the_limit(joint, sign):
    """gait_params (4 N.m motors, Bullet-order rows), limits at +-0.4 rad, a target of +-1.0 rad on one odd (yaw) joint, 200 raw
    ticks: the joint rests within 5 mrad of the limit, its motor is saturated (applied torque +-4 N.m) and limit rows were active.
    (An even joint would not do: with the same target the oracle leaves joint 2 near 0, so its limit rows never come into play.)"""
    o = Oracle(1, gait_params())
    o.set_joint_limits(True, 0.4)
    o.reset()
    tg = np.zeros((1, 16))
    tg[0, joint] = sign * 1.0
    o.tick(tg, 200)
    s = o.get_state()[0]
    q, tau = s[13 + joint], s[45 + joint]
    assert abs(abs(q) - 0.4) <= 5e-3 and np.sign(q) == sign, q
    assert abs(tau - sign * 4.0) <= 5e-4, tau
    assert o.row_stats()[1] > 0
    o.close()
