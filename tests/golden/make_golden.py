#!/usr/bin/env python3
"""Generate tests/golden/*.npz by running the reference's OWN Python task logic.

The unmodified ``/root/reference/SnakeGymEnv.py`` and ``/root/reference/snake.py`` are imported with
stub ``gym`` / ``pybullet`` / ``pybullet_data`` modules (SURVEY.md section 4, "a usable seam") and a fake
pybullet *client object* whose physics state is one environment of the CPU oracle.  Everything the
reference computes in Python -- clipping, createAction, the checkFeedback tick loop, the height
break, the 41-tick cap, getObservation packing, reward, termination, the in-step reset and the
SubprocVecEnv worker's second reset -- is therefore executed by the reference's code, and the
recorded (obs, reward, done, ticks) pin the oracle's and the CUDA kernel's restatement of rows
a1-a5, a8-a12, a15 of SURVEY.md section 8.  The physics tick underneath is the oracle's (PyBullet
itself is not installable here), so these vectors do NOT pin the tick against Bullet.

Run in the authoring container only (needs /root/reference):  python tests/golden/make_golden.py
"""
import os
import sys
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
REF = "/root/reference"

from oracle.oracle_py import Oracle  # noqa: E402
from bullet_envs_b200 import build_model, default_params  # noqa: E402


def install_stubs():
    gym = types.ModuleType("gym")

    class Env(object):
        pass

    class Box(object):
        def __init__(self, low, high):
            self.low, self.high, self.shape = np.asarray(low), np.asarray(high), np.asarray(low).shape

    gym.Env = Env
    gym.spaces = types.SimpleNamespace(Box=Box)
    sys.modules["gym"] = gym
    pb = types.ModuleType("pybullet")
    sys.modules["pybullet"] = pb
    pbd = types.ModuleType("pybullet_data")
    pbd.getDataPath = lambda: "/nonexistent"
    sys.modules["pybullet_data"] = pbd


class FakeClient:
    """The subset of the pybullet client API that snake.py calls, backed by one oracle environment."""
    URDF_USE_SELF_COLLISION = 8
    POSITION_CONTROL = 2

    def __init__(self, params=None, model=None):
        self.model = model or build_model()
        self.oracle = Oracle(1, params or default_params(), self.model)
        self.targets = np.zeros(16)
        self.ticks = 0
        self.calls = 0
        self.motor_of_joint = {j: i for i, j in enumerate(self.model.motor_joint_indices)}

    # world building: constant in the oracle
    def resetSimulation(self): self.calls += 1
    def setAdditionalSearchPath(self, p): self.calls += 1
    def setGravity(self, x, y, z): self.calls += 1
    def loadURDF(self, *a, **k): self.calls += 1; return 1
    def changeDynamics(self, *a, **k): self.calls += 1
    def enableJointForceTorqueSensor(self, *a, **k): self.calls += 1
    def getNumJoints(self, body): self.calls += 1; return self.model.num_urdf_joints

    def resetJointState(self, body, j, value):  # SURVEY A.6: q = value, qd = 0
        self.calls += 1
        s = self.oracle.get_state()
        m = self.motor_of_joint[j]
        s[0, 13 + m] = value
        s[0, 29 + m] = 0.0
        self.oracle.set_state(s)

    def resetBasePositionAndOrientation(self, body, pos, orn):  # pose set, base velocity zeroed
        self.calls += 1
        s = self.oracle.get_state()
        s[0, 0:3] = pos
        s[0, 3:7] = orn
        s[0, 7:13] = 0.0
        self.oracle.set_state(s)

    def getBasePositionAndOrientation(self, body):
        self.calls += 1
        s = self.oracle.get_state()[0]
        return tuple(s[0:3]), tuple(s[3:7])

    def getJointState(self, body, j):
        self.calls += 1
        s = self.oracle.get_state()[0]
        if j in self.motor_of_joint:
            m = self.motor_of_joint[j]
            return s[13 + m], s[29 + m], (0.0,) * 6, s[45 + m]
        if j == 0:  # fixed joint kdl_dummy_root -> base: only the reaction Fz is modelled
            return 0.0, 0.0, (0.0, 0.0, s[61], 0.0, 0.0, 0.0), 0.0
        return 0.0, 0.0, (0.0,) * 6, 0.0

    def getLinkStates(self, body, indices):
        self.calls += 1
        Rw, pw, _ = self.oracle.kinematics(0)
        out = []
        for li in indices:
            assert li % 3 == 0
            h = li // 3
            b = self.model.height_body[h]
            p = pw[b] + Rw[b] @ self.model.height_pt[h]
            out.append((tuple(p), (0, 0, 0, 1)))
        # Snake.getLinkPositions does np.array(data) on these ragged tuples (snake.py:143), which numpy >= 1.24
        # refuses; hand the same tuples back in the object array that older numpy built implicitly
        arr = np.empty((len(out), 2), dtype=object)
        for i, (p, q) in enumerate(out):
            arr[i, 0], arr[i, 1] = p, q
        return arr

    def setJointMotorControlArray(self, body, joints, mode, targetPositions=None, forces=None, **k):
        self.calls += 1
        assert mode == self.POSITION_CONTROL and list(joints) == self.model.motor_joint_indices
        assert all(np.isinf(f) for f in forces)
        self.targets = np.asarray(targetPositions, float)

    def stepSimulation(self):
        self.calls += 1
        self.ticks += 1
        self.oracle.tick(self.targets[None, :], 1)


def scenario_actions():
    rng = np.random.default_rng(2019)
    sc = {}
    sc["const_half"] = np.full((12, 8), 0.5)                       # test_script_env.py:16-17
    sc["random"] = rng.uniform(-1, 1, (40, 8))                      # PPO initial policy
    a = rng.uniform(-2.5, 2.5, (10, 8))                             # out-of-range -> checkBound clips in place
    sc["clipped"] = a
    t = np.arange(30)[:, None] * 0.3                                 # serpenoid on the odd joints (snake_gait_test.py:65-89)
    nn = (2 * np.arange(8) + 1)[None, :]
    sc["serpenoid"] = -np.sin(4 * nn + 2 * t)
    # joint 9 (action index 4) is held at its limit target pi/6 = 0.5236 > 0.5 while the other yaw joints swing: the tick loop
    # stops at |error|_2 <= 0.05, so joint 9 ends inside 0.5 when it carries the whole error (even steps: 0.476) and beyond it
    # when the others carry most of it (odd steps) -> `abs(observation[9]) > 0.5` fires (SnakeGymEnv.py:100), -5, double reset
    big = np.zeros((25, 8)); big[:, 4] = 1.0
    big[1::2, 0:4] = np.where(np.arange(12)[:, None] % 2 == 0, 1.0, -1.0)
    sc["terminate_q9"] = big
    # checkSnakeHeight (snake.py:237-245,299-301; SnakeGymEnv.py:99-103): the fake client's state is lifted before some steps
    # (see INJECT): 0 = dropped from z = 0.2 -> height break after the first tick; 3 = thrown upwards at 3 m/s from the ground
    # -> break in the middle of the tick loop; 5 = lifted with the action already reached -> zero ticks, done by checkTermination
    lift = np.zeros((8, 8)); lift[0] = 0.5; lift[1] = -0.5; lift[2] = 0.5; lift[3] = -0.7; lift[4] = 0.3; lift[5] = 0.3; lift[6] = 0.8; lift[7] = -0.2
    sc["lifted"] = lift
    return sc


# merged-body tables of a URDF that tests/test_model_tables.py compares between the reference's snake/snake.urdf and snake_chain.urdf
URDF_TABLES = ("joint_R0", "joint_t", "joint_axis", "joint_damping", "body_mass", "body_com", "body_inertia", "cyl_center", "cyl_axis",
               "cyl_fric_R", "cyl_radius", "cyl_halflen", "cyl_end", "cyl_break", "height_pt", "fz_axis", "cyl_body", "height_body")


def urdf_tables(path):
    m = build_model(path)
    out = {name: getattr(m, name) for name in URDF_TABLES}
    out["motor_joint_indices"] = np.asarray(m.motor_joint_indices)
    out["num_urdf_links"] = np.asarray(m.num_urdf_links)
    return out


# state edits applied to the (fake) simulator before a step: step -> (delta z of the base, delta vz of the base)
INJECT = {"lifted": {0: (0.2, 0.0), 3: (0.0, 3.0), 5: (0.2, 0.0)}}


def main():
    install_stubs()
    sys.path.insert(0, REF)
    time.sleep = lambda s: None  # Q2: the 10 ms wall-clock sleep per tick is not reproduced
    import snake as ref_snake
    import SnakeGymEnv as ref_env
    ref_snake.time.sleep = lambda s: None

    out = {}
    # both motor-row treatments of the oracle's tick: "" = the default (auto -> motor rows eliminated,
    # the kernel the reference configuration runs on), "pgs/" = Bullet-order rows inside the PGS
    for prefix, solver in (("", 2), ("pgs/", 0)):
      for name, actions in scenario_actions().items():
        name = prefix + name
        client = FakeClient(default_params(motor_solver=solver))
        robot = ref_snake.Snake(client, "snake/snake.urdf")
        env = ref_env.SnakeGymEnv(robot)
        obs0 = env.reset()                       # worker 'reset' command
        rec_obs, rec_rew, rec_done, rec_ticks, rec_act = [np.array(obs0)], [], [], [], []
        inj = np.zeros((len(actions), 2))
        for t, a in enumerate(actions):
            a_in = np.array(a, dtype=np.float64)
            if t in INJECT.get(name.split("/")[-1], {}):
                inj[t] = INJECT[name.split("/")[-1]][t]
                s = client.oracle.get_state(); s[0, 2] += inj[t, 0]; s[0, 9] += inj[t, 1]; client.oracle.set_state(s)
            t0 = client.ticks
            ob, r, d, info = env.step(a_in)      # may clip a_in in place
            if d:
                ob = env.reset()                 # ppo/multiprocessing_env.py:14-15
            rec_obs.append(np.array(ob)); rec_rew.append(float(r)); rec_done.append(bool(d))
            rec_ticks.append(client.ticks - t0); rec_act.append(a_in)
        out[name + "/actions"] = np.asarray(actions, np.float64)
        out[name + "/clipped_actions"] = np.asarray(rec_act)
        out[name + "/obs"] = np.asarray(rec_obs)
        out[name + "/rew"] = np.asarray(rec_rew)
        out[name + "/done"] = np.asarray(rec_done)
        out[name + "/ticks"] = np.asarray(rec_ticks, np.int32)
        out[name + "/inject"] = inj
        print("%-14s steps %3d  ticks/step %5.1f  dones %d  return %.4f  client calls %d" % (
            name, len(actions), np.mean(rec_ticks), int(np.sum(rec_done)), float(np.sum(rec_rew)), client.calls))
    out["meta/motor_list"] = np.asarray(robot.motorList)
    out["meta/obs_dim"] = np.asarray(env.observation_space.shape[0])
    out["meta/act_dim"] = np.asarray(env.action_space.shape[0])
    out["meta/obs_high"] = np.asarray(env.observation_space.high)
    path = os.path.join(ROOT, "tests", "golden", "reference_python_task_logic.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")

    # mode='test' info stream (snake.py:275-278,292-293; SnakeGymEnv.py:43-44): per-tick observations and link
    # positions recorded by the reference's own code; valid rows of all steps concatenated, `ticks` gives the split
    tm = {}
    for name in ("serpenoid", "terminate_q9"):
        actions = scenario_actions()[name][:14]
        client = FakeClient(default_params())
        robot = ref_snake.Snake(client, "snake/snake.urdf")
        env = ref_env.SnakeGymEnv(robot)
        robot.mode = env.mode = "test"
        env.reset()
        io, lp, tk, ob_l, rw, dn = [], [], [], [], [], []
        for a in actions:
            ob, r, d, info = env.step(np.array(a, dtype=np.float64))
            assert info["frames"] == [] and len(info["internal_observations"]) == len(info["link_positions"])
            tk.append(len(info["internal_observations"]))
            io += [np.asarray(x, np.float64) for x in info["internal_observations"]]
            lp += [np.asarray(x, np.float64) for x in info["link_positions"]]
            if d:
                ob = env.reset()
            ob_l.append(np.array(ob)); rw.append(float(r)); dn.append(bool(d))
        tm[name + "/actions"] = np.asarray(actions, np.float64)
        tm[name + "/ticks"] = np.asarray(tk, np.int32)
        tm[name + "/internal_observations"] = np.asarray(io).reshape(-1, 56)
        tm[name + "/link_positions"] = np.asarray(lp).reshape(-1, 51)
        tm[name + "/obs"] = np.asarray(ob_l); tm[name + "/rew"] = np.asarray(rw); tm[name + "/done"] = np.asarray(dn)
        print("test-mode %-14s steps %d ticks %d dones %d" % (name, len(actions), int(np.sum(tk)), int(np.sum(dn))))
    path = os.path.join(ROOT, "tests", "golden", "reference_python_test_mode.npz")
    np.savez_compressed(path, **tm)
    print("wrote", path, os.path.getsize(path), "bytes")

    # raw single-env use (no vector wrapper; a3c/agent.py:99-125 keeps stepping after `done`): SnakeGymEnv.step returns the
    # TERMINAL observation and the next step's reward uses the dead episode's x as x_prev (SURVEY Q8)
    raw = {}
    for name in ("serpenoid", "clipped"):
        actions = scenario_actions()[name]
        client = FakeClient(default_params())
        robot = ref_snake.Snake(client, "snake/snake.urdf")
        env = ref_env.SnakeGymEnv(robot)
        ob0 = env.reset()
        ob_l, rw, dn = [np.array(ob0)], [], []
        for a in actions:
            ob, r, d, info = env.step(np.array(a, dtype=np.float64))   # NO reset by the caller
            ob_l.append(np.array(ob)); rw.append(float(r)); dn.append(bool(d))
        raw[name + "/actions"] = np.asarray(actions, np.float64)
        raw[name + "/obs"] = np.asarray(ob_l); raw[name + "/rew"] = np.asarray(rw); raw[name + "/done"] = np.asarray(dn)
        print("raw single-env %-12s steps %d dones %d return %.4f" % (name, len(actions), int(np.sum(dn)), float(np.sum(rw))))
    path = os.path.join(ROOT, "tests", "golden", "reference_python_raw_single_env.npz")
    np.savez_compressed(path, **raw)
    print("wrote", path, os.path.getsize(path), "bytes")

    # the model tables PyBullet's importer would build from the reference's own URDF (snake.py:93)
    path = os.path.join(ROOT, "tests", "golden", "reference_urdf_model_tables.npz")
    np.savez_compressed(path, **urdf_tables(os.path.join(REF, "snake", "snake.urdf")))
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
