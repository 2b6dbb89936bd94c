"""Device-resident drop-in for the reference's vector environment.

:class:`SnakeVecEnv` keeps the interface of ``SubprocVecEnv`` (reference
``ppo/multiprocessing_env.py:31-153``: ``reset``, ``step``, ``step_async``/``step_wait``, ``close``,
``__len__``, ``num_envs``/``nenvs``, ``observation_space``, ``action_space``) but replaces the N
worker processes, pipes and PyBullet clients by one batch of N environments resident in HBM and one
CUDA kernel launch per ``step``.  Semantics are those of the worker loop (``:11-16``): on ``done``
the returned observation is the post-reset one.

* numpy actions in  -> numpy ``(obs[N,56], rews[N], dones[N] bool, infos)`` out, through the
  C-ABI ``snk_step_host`` (pinned H2D / D2H inside the library) -- the strict drop-in for
  ``ppo/train.py:122`` and ``ars/train.py:99``;
* CUDA torch actions in -> CUDA torch tensors out, zero-copy on the current torch stream; pass
  ``out=(obs, rew, done)`` to have the kernel write straight into rollout-buffer slices.

PyTorch is used for device memory and streams only.  There is no CPU fallback: constructing the
class without the CUDA extension or without a GPU raises.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _abi
from .spaces import Box
from .urdf_model import OBS_DIM, STATE_STRIDE, NJ, build_model

LINK_POS_DIM = 51  # SNK_LINK_POS_DIM: 17 links x (x, y, z), snake.py:138-146
MAN_STRIDE = 1056  # SNK_MAN_STRIDE: floats of contact cache per environment (32 cylinders x 4 slots x 8 words + 32 counts)


class SnakeVecEnv:
    def __init__(self, env_fns=None, num_envs=None, args=None, device=None, urdf_path=None, params=None,
                 model=None, obs_dtype=np.float64, pinned_io=False, mode=None):
        """``env_fns``: list of thunks as given to ``SubprocVecEnv`` (only its length is used -- the
        thunks would build PyBullet-backed envs) *or* pass ``num_envs``.  ``args``: the reference's
        argparse namespace (``ppo/params.py``) or None for the defaults.  ``device``: CUDA device
        index / ``torch.device``.  ``obs_dtype``: dtype of the numpy results (the reference returns float64;
        ``np.float32`` skips the conversion).  ``pinned_io``: the numpy path keeps persistent page-locked
        result buffers that the library uses as DMA targets directly; the arrays returned by ``step`` /
        ``reset`` are then views that stay valid until the next call (the reference's callers convert or
        consume them immediately: ``ppo/train.py:114,131-136``, ``ars/train.py:99-110``).  ``mode``: ``'train'``
        (default, or ``args.mode``) returns empty info dicts; ``'test'`` returns the reference's per-tick info stream
        (``SnakeGymEnv.py:43-44``): ``info['internal_observations']`` / ``info['link_positions']`` = one array per
        physics tick of the env-step (``snake.py:292-293``), ``info['frames']`` = [] (rendering needs a display)."""
        import torch

        if env_fns is not None and num_envs is None:
            num_envs = env_fns if isinstance(env_fns, int) else len(env_fns)
        if not num_envs or num_envs <= 0:
            raise ValueError("num_envs must be positive")
        self._torch = torch
        self._lib = _abi.load_library()
        if device is None:
            dev_index = torch.cuda.current_device() if torch.cuda.is_available() else 0
        else:
            d = torch.device(device) if not isinstance(device, int) else torch.device("cuda", device)
            dev_index = d.index if d.index is not None else 0
        self.device = torch.device("cuda", dev_index)
        self.params = params if params is not None else _abi.default_params(args)
        self.model = model if model is not None else build_model(urdf_path)
        self._cmodel = self.model.to_ctypes()
        self._h = ctypes.c_void_p()
        _abi.check(self._lib.snk_create(ctypes.byref(self._cmodel), ctypes.byref(self.params), int(num_envs), dev_index,
                                        ctypes.byref(self._h)), self._lib)
        self.num_envs = self.nenvs = int(num_envs)
        self.act_dim = int(self._lib.snk_action_dim(self._h))
        self.obs_dtype = obs_dtype
        self.waiting = False
        self.closed = False
        self._pending = None
        self._infos = tuple({} for _ in range(self.num_envs))  # SnakeGymEnv.py:45-46 (train mode)
        self.mode = mode if mode is not None else (getattr(args, "mode", "train") if args is not None else "train")
        self.max_ticks = int(self.params.max_ticks)
        # spaces: snake.py:166-177, SnakeGymEnv.py:60-79
        hi = np.zeros(OBS_DIM)
        hi[0:NJ] = np.pi
        hi[NJ:3 * NJ] = np.inf
        hi[3 * NJ:] = 1.0
        self.observation_space = Box(-hi, hi)
        self.action_space = Box(-np.ones(self.act_dim), np.ones(self.act_dim))
        self.last_ticks = None
        self._pin = None
        if pinned_io:
            pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True).numpy()
            self._pin = dict(act=pin((self.num_envs, self.act_dim), torch.float32), obs=pin((self.num_envs, OBS_DIM), torch.float32),
                             rew=pin((self.num_envs,), torch.float32), done=pin((self.num_envs,), torch.uint8),
                             ticks=pin((self.num_envs,), torch.int32))

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return ctypes.c_void_p(self._torch.cuda.current_stream(self.device).cuda_stream)

    @staticmethod
    def _ptr(t):
        return ctypes.c_void_p(t.data_ptr())

    def _check_open(self):
        if self.closed or not self._h:
            raise RuntimeError("SnakeVecEnv is closed")

    # ------------------------------------------------------------------ SubprocVecEnv surface
    def reset(self, mask=None, as_torch=False, hard=False):
        """Soft reset (``snake.py:119-127``) of all environments (or of ``mask``); returns obs [N,56].  ``hard=True`` is
        ``Snake.reset(hardReset=True)`` (``snake.py:88-95``): the world is rebuilt, so the applied-torque / reaction-force
        slots that a soft reset leaves stale (SURVEY Q9) read zero as well.  With persistent manifolds on (``set_manifold`` or
        ``set_bullet_tick``), the contact caches of the
        hard-reset environments are emptied too (a rebuilt world has no cached points; the caches survive SOFT resets only, Q10)."""
        self._check_open()
        torch = self._torch
        if hard:
            m = torch.ones(self.num_envs, dtype=torch.bool, device=self.device) if mask is None else \
                torch.as_tensor(np.asarray(mask) if not torch.is_tensor(mask) else mask, device=self.device).bool()
            if tuple(m.shape) != (self.num_envs,):
                raise ValueError("mask must have one entry per environment")
            st = self.get_state()
            st[m] = 0.0
            st[m, 6] = 1.0  # SNK_S_QUAT + 3
            self.set_state(st)
            if getattr(self, "_manifold", None) or getattr(self, "_bullet", None) is not None:
                mb = None if mask is None else m.to(torch.uint8).contiguous()
                _abi.check(self._lib.snk_clear_manifold(self._h, None if mb is None else self._ptr(mb), self._stream()), self._lib)
                torch.cuda.current_stream(self.device).synchronize()
        if as_torch or (mask is not None and torch.is_tensor(mask) and mask.is_cuda):
            obs = torch.empty((self.num_envs, OBS_DIM), dtype=torch.float32, device=self.device)
            m = None if mask is None else mask.to(device=self.device, dtype=torch.uint8).contiguous()
            _abi.check(self._lib.snk_reset(self._h, None if m is None else self._ptr(m), self._ptr(obs), self._stream()), self._lib)
            return obs
        obs = np.empty((self.num_envs, OBS_DIM), np.float32)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        _abi.check(self._lib.snk_reset_host(self._h, None if m is None else ctypes.c_void_p(m.ctypes.data),
                                            ctypes.c_void_p(obs.ctypes.data)), self._lib)
        return obs.astype(self.obs_dtype, copy=False)

    def _step_test_mode(self, actions, out):
        """mode='test' (snake.py:275-278,292-293): the step through ``snk_step_trace`` with the per-tick info stream."""
        torch = self._torch
        n, cuda_in = self.num_envs, torch.is_tensor(actions) and actions.is_cuda
        a = (actions if cuda_in else torch.as_tensor(np.ascontiguousarray(np.asarray(actions), np.float32), device=self.device))
        a = a.to(dtype=torch.float32).contiguous().view(n, self.act_dim)
        if out is None or not cuda_in:
            obs = torch.empty((n, OBS_DIM), dtype=torch.float32, device=self.device)
            rew = torch.empty((n,), dtype=torch.float32, device=self.device)
            done = torch.empty((n,), dtype=torch.uint8, device=self.device)
        else:
            obs, rew, done = out
        ticks = torch.empty((n,), dtype=torch.int32, device=self.device)
        tobs = torch.empty((n, self.max_ticks, OBS_DIM), dtype=torch.float32, device=self.device)
        tlnk = torch.empty((n, self.max_ticks, LINK_POS_DIM), dtype=torch.float32, device=self.device)
        _abi.check(self._lib.snk_step_trace(self._h, self._ptr(a), self._ptr(obs), self._ptr(rew), self._ptr(done), self._ptr(ticks),
                                            self._ptr(tobs), self._ptr(tlnk), self._stream()), self._lib)
        tk = ticks.cpu().numpy()
        tobs_h, tlnk_h = tobs.cpu().numpy().astype(self.obs_dtype), tlnk.cpu().numpy().astype(self.obs_dtype)
        infos = tuple({"frames": [], "internal_observations": [tobs_h[e, k] for k in range(tk[e])],
                       "link_positions": [tlnk_h[e, k] for k in range(tk[e])]} for e in range(n))
        if cuda_in:
            self._pending = ("torch", obs, rew, done, ticks, infos)
        else:
            self._pending = ("numpy", obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy(), tk, infos)
        self.waiting = True

    def step_async(self, actions, out=None):
        self._check_open()
        torch = self._torch
        if self.mode == "test":
            return self._step_test_mode(actions, out)
        if torch.is_tensor(actions) and actions.is_cuda:
            a = actions.to(dtype=torch.float32).contiguous().view(self.num_envs, self.act_dim)
            if out is None:
                obs = torch.empty((self.num_envs, OBS_DIM), dtype=torch.float32, device=self.device)
                rew = torch.empty((self.num_envs,), dtype=torch.float32, device=self.device)
                done = torch.empty((self.num_envs,), dtype=torch.uint8, device=self.device)
            else:
                obs, rew, done = out
                for t, shape, dt in ((obs, (self.num_envs, OBS_DIM), torch.float32), (rew, (self.num_envs,), torch.float32),
                                     (done, (self.num_envs,), torch.uint8)):
                    if not (t.is_cuda and t.is_contiguous() and t.dtype == dt and tuple(t.shape) == shape):
                        raise ValueError("out tensors must be contiguous CUDA tensors obs[N,56] f32, rew[N] f32, done[N] u8")
            ticks = torch.empty((self.num_envs,), dtype=torch.int32, device=self.device)
            _abi.check(self._lib.snk_step(self._h, self._ptr(a), self._ptr(obs), self._ptr(rew), self._ptr(done), self._ptr(ticks),
                                          self._stream()), self._lib)
            self._pending = ("torch", obs, rew, done, ticks, self._infos)
        else:
            if self._pin is not None:
                a = self._pin["act"]
                a[...] = np.asarray(actions).reshape(self.num_envs, self.act_dim)
                obs, rew, done, ticks = (self._pin[k] for k in ("obs", "rew", "done", "ticks"))
            else:
                f64 = np.dtype(self.obs_dtype) == np.float64  # the reference's dtypes: snk_step_host_f64 converts on its threads
                dt = np.float64 if f64 else np.float32
                a = np.ascontiguousarray(np.asarray(actions), dt).reshape(self.num_envs, self.act_dim)
                obs = np.empty((self.num_envs, OBS_DIM), dt)
                rew = np.empty(self.num_envs, dt)
                done = np.empty(self.num_envs, np.uint8)
                ticks = np.empty(self.num_envs, np.int32)
            p = lambda x: ctypes.c_void_p(x.ctypes.data)
            fn = self._lib.snk_step_host_f64 if obs.dtype == np.float64 else self._lib.snk_step_host
            _abi.check(fn(self._h, p(a), p(obs), p(rew), p(done), p(ticks)), self._lib)
            self._pending = ("numpy", obs, rew, done, ticks, self._infos)
        self.waiting = True

    def step_wait(self):
        if self._pending is None:
            raise RuntimeError("step_wait() without step_async()")
        kind, obs, rew, done, ticks, infos = self._pending
        self._pending = None
        self.waiting = False
        self.last_ticks = ticks
        if kind == "torch":
            return obs, rew, done.bool(), infos
        return obs.astype(self.obs_dtype, copy=False), rew.astype(self.obs_dtype, copy=False), done.view(np.bool_), infos

    def step(self, actions, out=None):
        self.step_async(actions, out=out)
        return self.step_wait()

    def close(self):
        if self.closed:
            return
        self.closed = True
        if self._h:
            self._lib.snk_destroy(self._h)
            self._h = None

    def __len__(self):
        return self.nenvs

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ extras (parity harness, gait script)
    def tick(self, targets, n_ticks=1):
        """Raw physics ticks with joint targets [N,16] (``snake_gait_test.py:96-104``)."""
        self._check_open()
        torch = self._torch
        t = torch.as_tensor(np.asarray(targets, np.float32) if not torch.is_tensor(targets) else targets, dtype=torch.float32,
                            device=self.device).contiguous().view(self.num_envs, NJ)
        _abi.check(self._lib.snk_tick(self._h, self._ptr(t), int(n_ticks), self._stream()), self._lib)
        torch.cuda.current_stream(self.device).synchronize()

    def rollout_linear(self, weights, n_steps, mean=None, inv_std=None, noise=None, trace=False):
        """``n_steps`` env-steps in one launch with a linear policy per environment (ARS rollouts,
        ``ars/train.py:74-116``): before every step ``action = W_env @ ((obs + noise[t]) - mean) * inv_std``.
        ``weights`` [N, act_dim, 56]; ``mean`` / ``inv_std`` [56] or None; ``noise`` [n_steps, N, 56] or None.
        Returns the per-environment sum of rewards (CUDA tensor) and, with ``trace=True``, every input the
        policy saw [n_steps, N, 56] for the caller's running statistics."""
        self._check_open()
        torch = self._torch
        dev = lambda x, shape: None if x is None else torch.as_tensor(x, dtype=torch.float32, device=self.device).contiguous().view(shape)
        w = dev(weights, (self.num_envs, self.act_dim, OBS_DIM))
        m, s = dev(mean, (OBS_DIM,)), dev(inv_std, (OBS_DIM,))
        z = dev(noise, (n_steps, self.num_envs, OBS_DIM))
        ret = torch.empty((self.num_envs,), dtype=torch.float32, device=self.device)
        tr = torch.empty((n_steps, self.num_envs, OBS_DIM), dtype=torch.float32, device=self.device) if trace else None
        p = lambda x: None if x is None else self._ptr(x)
        _abi.check(self._lib.snk_rollout_linear(self._h, p(w), p(m), p(s), p(z), int(n_steps), p(ret), p(tr), self._stream()), self._lib)
        return (ret, tr) if trace else ret

    def observe(self):
        torch = self._torch
        obs = torch.empty((self.num_envs, OBS_DIM), dtype=torch.float32, device=self.device)
        _abi.check(self._lib.snk_observe(self._h, self._ptr(obs), self._stream()), self._lib)
        return obs

    def self_clearance(self):
        """Lower bound [N] (metres, CUDA tensor) of the smallest distance between two non-consecutive cylinders of every
        environment -- the pairs ``URDF_USE_SELF_COLLISION`` (``snake.py:93``) makes Bullet test.  Positive over a run =
        no self-contact was missed (SURVEY.md Q11)."""
        torch = self._torch
        c = torch.empty((self.num_envs,), dtype=torch.float32, device=self.device)
        _abi.check(self._lib.snk_self_clearance(self._h, self._ptr(c), self._stream()), self._lib)
        return c

    def get_state(self):
        torch = self._torch
        s = torch.empty((self.num_envs, STATE_STRIDE), dtype=torch.float32, device=self.device)
        _abi.check(self._lib.snk_get_state(self._h, self._ptr(s), self._stream()), self._lib)
        return s

    def set_state(self, state):
        torch = self._torch
        s = torch.as_tensor(state, dtype=torch.float32, device=self.device).contiguous().view(self.num_envs, STATE_STRIDE)
        _abi.check(self._lib.snk_set_state(self._h, self._ptr(s), self._stream()), self._lib)
        torch.cuda.current_stream(self.device).synchronize()

    def state_dict(self):
        """Checkpoint of the whole batch (the reference never checkpoints simulator state; SURVEY.md section 5):
        the [N,64] state array on the CPU plus the parameters' bytes.  With persistent manifolds on, also their warm-start
        factor (``manifold_warm``) and contact caches (``manifold_cache``, [N,1056] on the CPU), so that a restored batch
        continues bit for bit.  With Bullet's literal tick on, ``bullet_tick_warm`` and the caches (``manifold_cache``).  With the
        joint-limit rows on, their angle (``joint_limit_angle``)."""
        sd = {"state": self.get_state().cpu(), "num_envs": self.num_envs, "params": bytes(self.params)}
        if getattr(self, "_manifold", None):
            sd["manifold_warm"] = self._manifold[1]
            sd["manifold_cache"] = self.get_manifold_cache().cpu()
        if getattr(self, "_bullet", None) is not None:
            sd["bullet_tick_warm"] = self._bullet
            sd["manifold_cache"] = self.get_manifold_cache().cpu()
        if getattr(self, "_limits", None) is not None:
            sd["joint_limit_angle"] = self._limits
        return sd

    def _contact_model(self):
        if getattr(self, "_bullet", None) is not None:
            return ("Bullet tick", self._bullet)
        if getattr(self, "_manifold", None):
            return ("persistent manifolds", self._manifold[1])
        return ("default", None)

    def load_state_dict(self, sd):
        """Restore a :meth:`state_dict`.  Raises ``ValueError`` when the checkpoint comes from a batch with another size, other
        parameters, another contact model (default, persistent manifolds, Bullet's literal tick, or another warm-start factor) or
        another joint-limit setting (off, or another angle); nothing is touched then."""
        if int(sd["num_envs"]) != self.num_envs or bytes(sd["params"]) != bytes(self.params):
            raise ValueError("checkpoint was taken from a batch with another size or other parameters")
        mine = self._contact_model()
        theirs = ("Bullet tick", float(sd["bullet_tick_warm"])) if "bullet_tick_warm" in sd else \
            ("persistent manifolds", float(sd["manifold_warm"])) if "manifold_warm" in sd else ("default", None)
        if mine != theirs:
            fmt = lambda m: m[0] if m[1] is None else "%s, warm %g" % m
            raise ValueError("checkpoint was taken with another contact model (%s; this batch: %s)" % (fmt(theirs), fmt(mine)))
        lim_mine = getattr(self, "_limits", None)
        lim_theirs = float(sd["joint_limit_angle"]) if "joint_limit_angle" in sd else None
        if lim_mine != lim_theirs:
            fmt = lambda a: "off" if a is None else "+-%g rad" % a
            raise ValueError("checkpoint was taken with other joint limits (%s; this batch: %s)" % (fmt(lim_theirs), fmt(lim_mine)))
        if mine[1] is not None:
            self.set_manifold_cache(sd["manifold_cache"])  # checked before anything is touched
        self.set_state(sd["state"])

    def set_manifold(self, on=True, warm=0.1):
        """Bullet's persistent contact manifolds + contact warm starting (``snk_set_manifold``; SURVEY.md 8f rank 2): 4 cached points
        per cylinder fed by the hull's support vertex, normal impulses of the previous tick x ``warm``.  Clears the caches.  Mirrors
        the oracle's ``Oracle.set_manifold``; the default (off) is the one-point-per-cylinder tick the benchmark runs."""
        _abi.check(self._lib.snk_set_manifold(self._h, int(bool(on)), float(warm)), self._lib)
        self._manifold = (True, float(warm)) if on else None

    def set_bullet_tick(self, on=True, warm=0.1):
        """Bullet's literal tick (``snk_set_bullet_tick``): Bullet-order motor rows relaxed in the PGS together with the persistent
        manifolds and warm starting (x ``warm``) -- stepSimulation's own tick, on any handle.  Clears the caches; ``on=False`` returns
        to the handle's own solver.  Mirrors the oracle twin ``BulletTickOracle.set_bullet_tick`` (tests/); ``rollout_linear`` is refused while it is on."""
        _abi.check(self._lib.snk_set_bullet_tick(self._h, int(bool(on)), float(warm)), self._lib)
        self._bullet = float(warm) if on else None

    def set_joint_limits(self, on=True, angle=1.57):
        """Joint-limit rows (``snk_set_joint_limits``; PyBullet's btMultiBodyJointLimitConstraint, which loadURDF gives every
        revolute joint of snake.urdf at +-1.57 rad): two unilateral rows per joint at +-``angle``, solved after the motor rows in
        every sweep.  For the kernels with Bullet-order motor rows: ``motor_solver=0`` (or auto with a finite motor force) and
        Bullet's literal tick (``set_bullet_tick``).  Refused on a handle with the exact motor solver unless the Bullet tick is on.
        Off by default; mirrors ``Oracle.set_joint_limits``."""
        self._check_open()
        _abi.check(self._lib.snk_set_joint_limits(self._h, int(bool(on)), float(angle)), self._lib)
        self._limits = float(angle) if on else None

    def joint_limit_stats(self):
        """(limit rows active at the end of a tick, summed over the environments and ticks of the last step launch, those ticks) --
        ``snk_joint_limit_stats``; the oracle's ``row_stats()[1]`` counts the same rows."""
        out = (ctypes.c_int64 * 2)()
        _abi.check(self._lib.snk_joint_limit_stats(self._h, out), self._lib)
        return int(out[0]), int(out[1])

    def get_manifold_cache(self):
        """The persistent manifolds' contact caches as a CUDA tensor [N, 1056] (``snk_get_manifold_cache``; layout in
        include/snake_b200.h at SNK_MAN_STRIDE)."""
        self._check_open()
        torch = self._torch
        c = torch.empty((self.num_envs, MAN_STRIDE), dtype=torch.float32, device=self.device)
        _abi.check(self._lib.snk_get_manifold_cache(self._h, self._ptr(c), self._stream()), self._lib)
        return c

    def set_manifold_cache(self, cache):
        """Load contact caches [N, 1056] (``snk_set_manifold_cache``).  Raises when a point count is not an integer in 0..4; the
        caches are then left as they were."""
        self._check_open()
        torch = self._torch
        c = torch.as_tensor(cache, dtype=torch.float32, device=self.device).contiguous()
        if tuple(c.shape) != (self.num_envs, MAN_STRIDE):
            raise ValueError("manifold cache must be [%d, %d]" % (self.num_envs, MAN_STRIDE))
        _abi.check(self._lib.snk_set_manifold_cache(self._h, self._ptr(c), self._stream()), self._lib)
        torch.cuda.current_stream(self.device).synchronize()

    def manifold_stats(self):
        """(cached contact points summed over the ticks of the last step launch, ticks) -- ``snk_manifold_stats``."""
        out = (ctypes.c_int64 * 2)()
        _abi.check(self._lib.snk_manifold_stats(self._h, out), self._lib)
        return int(out[0]), int(out[1])

    def counters(self):
        """Device counters of the last step launch: ticks, PGS iterations, dones, non-finite resets."""
        out = (ctypes.c_int64 * 4)()
        _abi.check(self._lib.snk_last_counters(self._h, out), self._lib)
        return dict(ticks=out[0], pgs_iterations=out[1], dones=out[2], nonfinite=out[3])

    def launch_count(self):
        return int(self._lib.snk_launch_count(self._h))
