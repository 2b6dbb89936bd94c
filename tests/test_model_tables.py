"""URDF -> merged tables (SURVEY.md section 8a, "model facts")."""
import os

import numpy as np
import pytest

from bullet_envs_b200.urdf_model import DEFAULT_URDF, ImportRules, build_model, dfs_order, parse_urdf

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_urdf_model_tables.npz")


def test_link_and_joint_counts_and_motor_indices(model):
    links, joints = parse_urdf(DEFAULT_URDF)
    assert len(links) == 50 and len(joints) == 49
    assert sum(j.jtype == "revolute" for j in joints) == 16 and sum(j.jtype == "fixed" for j in joints) == 33
    root, order = dfs_order(links, joints)
    assert root == "kdl_dummy_root" and order[0].child == "base"
    # Snake.buildMotorList: motorList = arange(3, numJoints, 3)  (snake.py:78-81)
    assert model.motor_joint_indices == list(range(3, 49, 3))
    assert [order[i].jtype for i in model.motor_joint_indices] == ["revolute"] * 16


def test_masses_follow_bullet_import_rules(model):
    # no <inertial> => mass 1 (root, base, 16 collars): 3.296 kg of file masses + 18 kg
    assert model.body_mass.sum() == pytest.approx(21.296, abs=1e-9)
    assert model.body_mass[0] == pytest.approx(3.103) and model.body_mass[16] == pytest.approx(0.103)
    assert np.allclose(model.body_mass[1:16], 1.206)
    plain = build_model(rules=ImportRules(unit_mass_for_missing_inertial=False, inertia_from_collision_aabb=False))
    assert plain.body_mass.sum() == pytest.approx(3.296, abs=1e-9)
    # inertia from file survives the merge when requested
    assert plain.body_inertia[16].reshape(3, 3)[2, 2] == pytest.approx(3.4814e-5)
    # default: AABB box of the 32-gon hull + 0.001 margin (SURVEY A.1): (3.55e-5, 3.55e-5, 5.01e-5)
    I16 = model.body_inertia[16].reshape(3, 3)
    assert np.allclose(np.diag(I16), [0.103 / 12 * (0.054 ** 2 + 0.035 ** 2)] * 2 + [0.103 / 12 * 2 * 0.054 ** 2], rtol=1e-9)


def test_zero_pose_geometry(model):
    from oracle.oracle_py import Oracle
    o = Oracle(1, model=model)
    o.reset()
    Rw, pw, height = o.kinematics(0)
    k = np.arange(1, 17)
    assert np.allclose(pw[1:, 0], -(0.0366 + 0.0639 * (k - 1)), atol=1e-9)   # chain laid along world -x
    assert np.allclose(pw[1:, 2], 0.026, atol=2e-5)                           # at cylinder-radius height
    assert pw[16, 0] == pytest.approx(-0.9951, abs=1e-9)
    assert height == pytest.approx(0.026, abs=1e-5)
    # consecutive joint axes alternate: even motors pitch (axis ~ world y), odd motors yaw (axis ~ world z)
    for i in range(16):
        a = Rw[i + 1] @ model.joint_axis[i]
        assert abs(a[1 if i % 2 == 0 else 2]) > 0.999


def test_cylinders_and_contact_rims(model):
    assert len(model.cyl_body) == 32
    counts = np.bincount(model.cyl_body, minlength=17)
    assert counts[0] == 1 and counts[16] == 1 and (counts[1:16] == 2).all()
    assert np.allclose(model.cyl_radius, 0.026) and np.allclose(model.cyl_halflen, 0.0165)
    # every cylinder's contact rim is the end that is an extreme of its merged body
    for b in range(1, 16):
        idx = np.where(model.cyl_body == b)[0]
        z = [model.cyl_center[i] @ model.cyl_axis[i] + model.cyl_end[i] * model.cyl_halflen[i] for i in idx]
        assert sorted(np.round(z, 4)) == [0.0018, 0.0621]
    # anisotropy anchor (SURVEY A.5): module 1 local (x,y,z) = world (+z,+y,-x); module 2 = (-y,+z,-x)
    R1 = model.cyl_fric_R[0].reshape(3, 3)   # body 0 frame == world at the zero pose
    assert np.allclose(R1, [[0, 0, -1], [0, 1, 0], [1, 0, 0]], atol=1e-9)


def test_height_points_and_fz_axis(model):
    assert list(model.height_body) == list(range(17))
    assert np.allclose(model.height_pt[0], [0, 0, 0.026]) and np.allclose(model.height_pt[1:], 0)
    assert np.allclose(model.fz_axis, [-1, 0, 0], atol=1e-9) and model.root_mass == 1.0


def test_generated_urdf_equals_reference_urdf(model):
    """the tables of the physics-only snake_chain.urdf against those of the reference's snake/snake.urdf, stored by
    tests/golden/make_golden.py (urdf_tables)"""
    ref = np.load(GOLDEN)
    names = ("joint_R0", "joint_t", "joint_axis", "joint_damping", "body_mass", "body_com", "body_inertia", "cyl_center",
             "cyl_axis", "cyl_fric_R", "cyl_radius", "cyl_halflen", "cyl_end", "cyl_break", "height_pt", "fz_axis", "cyl_body",
             "height_body")
    assert sorted(ref.files) == sorted(names + ("motor_joint_indices", "num_urdf_links"))
    for name in names:
        assert np.array_equal(ref[name], getattr(model, name)), name
    assert list(ref["motor_joint_indices"]) == model.motor_joint_indices and int(ref["num_urdf_links"]) == 50


def test_ctypes_round_trip(model):
    cm = model.to_ctypes()
    assert np.allclose(np.frombuffer(cm.joint_t, np.float64).reshape(16, 3), model.joint_t)
    assert list(cm.cyl_body) == list(model.cyl_body) and cm.root_mass == 1.0
