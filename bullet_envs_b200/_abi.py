"""ctypes mirror of ``include/snake_b200.h`` and the loader of the CUDA shared library.

The product path has no CPU fallback: if ``libsnake_b200.so`` is missing or a CUDA device is
absent, :func:`load_library` / ``snk_create`` raise and the caller fails loudly.
"""
from __future__ import annotations

import ctypes
import math
import os

from .urdf_model import CModel  # noqa: F401  (re-exported)

_HERE = os.path.dirname(os.path.abspath(__file__))
# SNK_B200_LIB points at another build of the same library (compile-variant A/B runs); the default is the in-tree build
LIB_PATH = os.environ.get("SNK_B200_LIB") or os.path.join(_HERE, "csrc", "libsnake_b200.so")


class CParams(ctypes.Structure):
    """ctypes mirror of ``snk_params``."""
    _fields_ = [
        ("dt", ctypes.c_double), ("gravity", ctypes.c_double * 3),
        ("motor_kp", ctypes.c_double), ("motor_kd", ctypes.c_double), ("motor_max_force", ctypes.c_double),
        ("scaling_factor", ctypes.c_double),
        ("alpha", ctypes.c_double), ("beta", ctypes.c_double), ("gamma", ctypes.c_double),
        ("energy_dt", ctypes.c_double), ("friction", ctypes.c_double), ("aniso", ctypes.c_double * 3),
        ("lin_damping", ctypes.c_double), ("ang_damping", ctypes.c_double),
        ("erp2", ctypes.c_double), ("linear_slop", ctypes.c_double), ("residual_threshold", ctypes.c_double),
        ("max_coord_vel", ctypes.c_double), ("err_threshold", ctypes.c_double), ("height_threshold", ctypes.c_double),
        ("term_angle", ctypes.c_double), ("done_penalty", ctypes.c_double),
        ("collision_force", ctypes.c_double), ("collision_penalty", ctypes.c_double),
        ("solver_iterations", ctypes.c_int32), ("max_ticks", ctypes.c_int32), ("gait_selection", ctypes.c_int32),
        ("cone_friction", ctypes.c_int32), ("term_joint", ctypes.c_int32), ("stale_obs_on_reset", ctypes.c_int32),
        ("alternate_motor_order", ctypes.c_int32), ("motor_solver", ctypes.c_int32),
    ]


def default_params(args=None, **overrides) -> CParams:
    """Reference defaults (``snake.py:8-9,25-27,55-64``; ``SnakeGymEnv.py:7-18``; SURVEY.md A.2).

    ``args`` may be the reference's argparse namespace (``ppo/params.py``): ``alpha``, ``beta``,
    ``gamma``, ``gaitSelection`` and ``scaling_factor`` are honoured exactly as ``Snake.setParams``
    / ``SnakeGymEnv.__init__`` do; ``kp``/``kd``/``motorTorqueLimit`` are ignored because the
    reference never passes them to PyBullet on the step path (SURVEY.md Q3/Q4)."""
    p = CParams()
    p.dt = 1.0 / 240.0
    p.gravity[:] = [0.0, 0.0, -9.8]
    p.motor_kp, p.motor_kd, p.motor_max_force = 0.1, 1.0, math.inf
    p.scaling_factor = math.pi / 6
    p.alpha, p.beta, p.gamma = 1.0, 0.01, 0.1
    p.energy_dt = 0.01
    p.friction = 2.0
    p.aniso[:] = [1.0, 0.1, 0.01]
    p.lin_damping = p.ang_damping = 0.04
    p.erp2, p.linear_slop, p.residual_threshold = 0.08, 1e-5, 1e-7
    p.max_coord_vel = 100.0
    p.err_threshold, p.height_threshold, p.term_angle = 0.05, 0.1, 0.5
    p.done_penalty, p.collision_force, p.collision_penalty = -5.0, 10.0, -10.0
    p.solver_iterations, p.max_ticks, p.gait_selection = 50, 41, 1
    p.cone_friction, p.term_joint, p.stale_obs_on_reset, p.alternate_motor_order = 1, 9, 1, 1
    p.motor_solver = 2  # auto: motor rows eliminated exactly when force = inf and kd = 1 (the reference's setting)
    if args is not None:
        p.alpha, p.beta, p.gamma = float(args.alpha), float(args.beta), float(args.gamma)
        p.gait_selection = int(args.gaitSelection)
        p.scaling_factor = math.pi / (float(args.scaling_factor) * 1.0)
    for k, v in overrides.items():
        if k in ("gravity", "aniso"):
            getattr(p, k)[:] = list(v)
        else:
            if not hasattr(p, k):
                raise AttributeError("unknown snk_params field %r" % k)
            setattr(p, k, v)
    return p


def gait_params(**overrides) -> CParams:
    """Physics settings of the open-loop gait script (``snake_gait_test.py:50-53,96``; SURVEY Q12):
    dt 0.01, g -9.81, motor force limit 4 N.m."""
    kw = dict(dt=0.01, gravity=[0.0, 0.0, -9.81], motor_max_force=4.0)
    kw.update(overrides)
    return default_params(**kw)


_lib = None


def load_library():
    """Load ``libsnake_b200.so`` (built in-tree by ``__graft_entry__.build()``) and type its ABI."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("CUDA extension %s is missing -- run `python __graft_entry__.py build`; "
                           "there is no CPU fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
    P = ctypes.POINTER
    lib.snk_default_params.argtypes = [P(CParams)]
    lib.snk_create.argtypes = [P(CModel), P(CParams), i64, ctypes.c_int, P(vp)]
    lib.snk_destroy.argtypes = [vp]
    lib.snk_num_envs.argtypes = [vp]; lib.snk_num_envs.restype = i64
    lib.snk_action_dim.argtypes = [vp]
    lib.snk_device.argtypes = [vp]
    lib.snk_reset.argtypes = [vp, vp, vp, vp]
    lib.snk_step.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    lib.snk_step_trace.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.snk_step_host.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.snk_step_host_f64.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.snk_reset_host.argtypes = [vp, vp, vp]
    lib.snk_tick.argtypes = [vp, vp, i32, vp]
    lib.snk_rollout_linear.argtypes = [vp, vp, vp, vp, vp, i32, vp, vp, vp]
    lib.snk_set_manifold.argtypes = [vp, ctypes.c_int, ctypes.c_double]
    lib.snk_manifold_stats.argtypes = [vp, P(i64)]
    lib.snk_get_manifold_cache.argtypes = [vp, vp, vp]
    lib.snk_set_manifold_cache.argtypes = [vp, vp, vp]
    lib.snk_clear_manifold.argtypes = [vp, vp, vp]
    lib.snk_gae.argtypes = [ctypes.c_int, vp, vp, vp, vp, ctypes.c_double, ctypes.c_double, vp, vp, i32, i64, vp]
    lib.snk_observe.argtypes = [vp, vp, vp]
    lib.snk_self_clearance.argtypes = [vp, vp, vp]
    lib.snk_get_state.argtypes = [vp, vp, vp]
    lib.snk_set_state.argtypes = [vp, vp, vp]
    lib.snk_last_counters.argtypes = [vp, P(i64)]
    lib.snk_launch_count.argtypes = [vp]; lib.snk_launch_count.restype = i64
    lib.snk_last_error.restype = ctypes.c_char_p
    lib.snk_build_info.restype = ctypes.c_char_p
    lib.snk_kernel_variant.restype = ctypes.c_char_p
    _lib = lib
    return lib


def check(rc, lib=None):
    if rc != 0:
        lib = lib or load_library()
        raise RuntimeError("snake_b200: %s (code %d)" % (lib.snk_last_error().decode(), rc))
