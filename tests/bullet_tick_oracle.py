"""ctypes front-end of the oracle with Bullet's literal tick (tests/oracle_bt/bullet_tick_oracle.c).  TEST INFRASTRUCTURE ONLY.

``BulletTickOracle`` is ``oracle.oracle_py.Oracle`` plus ``set_bullet_tick``: the library includes the oracle unchanged and adds the
composed tick, so every other method runs the oracle's own code."""
import ctypes
import os
import subprocess

from oracle.oracle_py import Oracle

_HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_bt")
SRC = os.path.join(_HERE, "bullet_tick_oracle.c")
ORACLE_SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "snake_oracle.c")
LIB = os.path.join(_HERE, "_build", "libbullet_tick_oracle.so")
CFLAGS = ["-O2", "-fPIC", "-std=gnu99", "-Wall", "-Wno-unused-function", "-ffp-contract=off"]   # those of oracle/Makefile


def build(force=False):
    """Compile the fp64 and fp32 builds into one library (the oracle's compiler flags)."""
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(SRC), os.path.getmtime(ORACLE_SRC)):
        out = os.path.dirname(LIB)
        os.makedirs(out, exist_ok=True)
        cc = os.environ.get("CC", "gcc")
        objs = []
        for tag, extra in (("f64", []), ("f32", ["-DSNK_REAL_FLOAT"])):
            o = os.path.join(out, "bt_%s.o" % tag)
            subprocess.check_call([cc] + CFLAGS + extra + ["-c", SRC, "-o", o])
            objs.append(o)
        subprocess.check_call([cc, "-shared", "-o", LIB] + objs + ["-lm"])
    return LIB


_lib = []


def _load():
    if not _lib:
        build()
        _lib.append(ctypes.CDLL(LIB))
    return _lib[0]


class BulletTickOracle(Oracle):
    """The oracle with ``set_bullet_tick``: while it is on, ``step`` / ``step_trace`` / ``tick`` run Bullet's literal tick."""

    _BT = {"step": "bt_step", "step_range": "bt_step_range", "step_trace": "bt_step_trace", "tick": "bt_tick"}

    def __init__(self, *args, **kw):
        self._bt_on = False
        super().__init__(*args, **kw)

    def _fn(self, name):
        return getattr(_load(), self.pfx + self._BT.get(name, name))

    def set_bullet_tick(self, on=True, warm=0.1):
        """Bullet's literal tick: the Bullet-order tick (motor rows relaxed in the PGS, whatever ``motor_solver`` the oracle was created
        with) on the contact set of the persistent manifolds, normal impulses warm-started x ``warm``.  Clears the caches;
        ``on=False`` restores the oracle's own tick.  Refused while ``set_manifold`` is on."""
        f = self._fn("bt_set"); f.restype = ctypes.c_int; f.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_double]
        if f(self._h, int(bool(on)), float(warm)) != 0:
            raise ValueError("set_bullet_tick refused (warm < 0, or persistent manifolds of the exact tick are on)")
        self._bt_on = bool(on)

    def set_manifold(self, on=True, warm=0.0):
        if self._bt_on:
            raise RuntimeError("set_manifold: Bullet's literal tick is on (set_bullet_tick); switch it off first")
        super().set_manifold(on, warm)
