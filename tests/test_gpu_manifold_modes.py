"""Persistent contact manifolds beyond snk_step (csrc/snake_manifold.cuh): the traced step (mode='test'), the fused linear-policy
rollout (snk_rollout_linear), the contact caches as state (snk_get/set_manifold_cache, checkpoints), masked hard resets
(snk_clear_manifold), and the release of the manifold memory by snk_destroy.

The oracle comparisons run freely from the reset pose.  The fp32 build of the oracle separates from the fp64 one at this rate
(measured on the CPU with the same inputs): first traced env-step of 128 environments, warm 0 and 0.1 -- tick counts identical,
joints 9e-8, link positions median (over environments of the largest error over ticks and links) 2.6e-5, largest 4.7e-3; rollout
of 192 environments x 3 steps, warm 0.1 -- ticks 14 933 vs 14 914, dones 80 vs 91, median return difference 6.0e-3.  The bounds
below are those with head room."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from bullet_envs_b200 import SnakeVecEnv, default_params

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STRIDE = 1056   # SNK_MAN_STRIDE
COUNTS = 1024   # first count word of an environment's cache row


@pytest.fixture(scope="module")
def torch():
    import torch as t
    if not t.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU fallback)")
    return t


def manifold_env(n, warm=0.1, mode=None):
    env = SnakeVecEnv(num_envs=n, device=0, mode=mode)
    env.set_manifold(True, warm)
    env.reset(as_torch=True)
    return env


def actions(torch, steps, n, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand((steps, n, 8), generator=g) * 2 - 1).cuda()


@pytest.mark.gpu
def test_traced_step_equals_the_step(torch):
    """snk_man_step_trace_kernel is the step with the per-tick info stream: the same bits for obs / rew / done / ticks, the caches
    and the counters; one info row per tick, the last one being the returned observation where the episode did not end."""
    n = 512
    acts = actions(torch, 4, n, 21)
    a, b = manifold_env(n), manifold_env(n, mode="test")
    rows = 0
    for t in range(4):
        oa, ra, da, _ = a.step(acts[t]); ca, sa = a.counters(), a.manifold_stats()
        ob, rb, db, info = b.step(acts[t]); cb, sb = b.counters(), b.manifold_stats()
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db) and torch.equal(a.last_ticks, b.last_ticks)
        assert torch.equal(a.get_manifold_cache(), b.get_manifold_cache())
        assert ca == cb and sa == sb and sa[0] > 0
        tk, dn, obn = b.last_ticks.cpu().numpy(), db.cpu().numpy(), ob.cpu().numpy()
        for e in range(n):
            assert len(info[e]["internal_observations"]) == tk[e] == len(info[e]["link_positions"])
            if tk[e] and not dn[e]:
                assert np.array_equal(info[e]["internal_observations"][-1].astype(np.float32), obn[e])
                rows += 1
    assert rows > n  # most env-steps took ticks and did not end
    a.close(); b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("warm", [0.0, 0.1])
def test_traced_step_vs_oracle(torch, warm):
    from oracle.oracle_py import Oracle
    n = 128
    acts = np.random.default_rng(31).uniform(-1, 1, (n, 8))
    o = Oracle(n, default_params()); o.set_manifold(True, warm); o.reset()
    _, _, _, ot, otobs, otlnk = o.step_trace(acts)
    env = manifold_env(n, warm, mode="test")
    _, _, _, info = env.step(torch.from_numpy(acts.astype(np.float32)).cuda())
    tk = env.last_ticks.cpu().numpy()
    assert (tk == ot).mean() >= 0.99, (tk == ot).mean()
    jmax, lerr = 0.0, []
    for e in np.nonzero(tk == ot)[0]:
        if tk[e] == 0:
            continue
        go, gl = np.stack(info[e]["internal_observations"]), np.stack(info[e]["link_positions"])
        jmax = max(jmax, np.abs(go[:, :16] - otobs[e, :tk[e], :16]).max())
        lerr.append(np.abs(gl - otlnk[e, :tk[e]]).max())
    assert len(lerr) > n // 2
    assert jmax < 1e-5, jmax                                          # joints follow the motor law
    assert np.median(lerr) < 5e-4 and max(lerr) < 5e-2, (np.median(lerr), max(lerr))   # link positions: contact sensitive
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1024, 40000])
def test_manifold_rollout_equals_the_stepwise_loop(torch, n):
    """Weights with a single non-zero per action row make the policy one exact product, so the fused rollout and
    `for t: env.step(policy(obs))` agree bit for bit.  40 000 environments are more than the 37 888 threads of the manifold grid on a
    B200 (148 SMs x 2 x 128), so threads take further environments from the global counter."""
    T = 4
    g = torch.Generator().manual_seed(2)
    noise = torch.rand((T, n, 56), generator=g).cuda()
    cols = torch.tensor([33, 1, 17, 49, 9, 55, 3, 20])
    gain = torch.rand((n, 8), generator=g) * 4 - 2
    W = torch.zeros((n, 8, 56)); W[:, torch.arange(8), cols] = gain
    W, gain, cols = W.cuda(), gain.cuda(), cols.cuda()
    fused = manifold_env(n)
    ret, trace = fused.rollout_linear(W, T, noise=noise, trace=True)
    cf, sf = fused.counters(), fused.manifold_stats()
    step = SnakeVecEnv(num_envs=n, device=0); step.set_manifold(True, 0.1)
    obs = step.reset(as_torch=True)
    acc = torch.zeros(n, device="cuda")
    ticks = iters = dones = pts = 0
    for t in range(T):
        x = obs + noise[t]
        assert torch.equal(x, trace[t])
        obs, rew, done, _ = step.step(gain * x[:, cols])
        acc += rew
        c = step.counters(); ticks += c["ticks"]; iters += c["pgs_iterations"]; dones += c["dones"]; pts += step.manifold_stats()[0]
    assert torch.equal(acc, ret)
    assert torch.equal(fused.get_state(), step.get_state())
    assert torch.equal(fused.get_manifold_cache(), step.get_manifold_cache())
    assert (cf["ticks"], cf["pgs_iterations"], cf["dones"], sf) == (ticks, iters, dones, (pts, ticks))
    assert ticks > n * T                                      # the rollout really moved
    fused.close(); step.close()


@pytest.mark.gpu
def test_manifold_rollout_vs_oracle(torch):
    from oracle.oracle_py import Oracle
    n, T = 192, 3
    rng = np.random.default_rng(8)
    W = (rng.normal(size=(n, 8, 56)) * 0.05).astype(np.float32)
    noise = rng.uniform(0, 1, (T, n, 56)).astype(np.float32)
    mean = rng.uniform(0.3, 0.7, 56).astype(np.float32); inv_std = rng.uniform(1.0, 3.0, 56).astype(np.float32)
    env = manifold_env(n)
    ret, tr = env.rollout_linear(W, T, mean=mean, inv_std=inv_std, noise=noise, trace=True)
    o = Oracle(n, default_params()); o.set_manifold(True, 0.1); o.reset()
    oret, otr = o.rollout_linear(W, T, mean=mean, inv_std=inv_std, noise=noise, trace=True)
    assert np.abs(tr[0].cpu().numpy() - otr[0]).max() < 1e-6   # first policy input: reset observation + noise
    c, oc = env.counters(), o.counters()
    assert abs(c["ticks"] - oc["ticks"]) <= 0.02 * oc["ticks"], (c, oc)
    assert abs(c["dones"] - oc["dones"]) <= 0.25 * oc["dones"] + 5, (c, oc)
    d = np.abs(ret.cpu().numpy() - oret)
    assert np.median(d) < 2e-2 and np.isfinite(ret.cpu().numpy()).all(), np.median(d)
    env.close()


@pytest.mark.gpu
def test_checkpoint_resumes_bit_exactly_with_manifolds(torch):
    n = 1024
    acts = actions(torch, 6, n, 13)
    a = manifold_env(n)
    for t in range(3):
        a.step(acts[t])
    sd = a.state_dict()
    assert sd["manifold_warm"] == 0.1 and tuple(sd["manifold_cache"].shape) == (n, STRIDE) and not sd["manifold_cache"].is_cuda
    b = SnakeVecEnv(num_envs=n, device=0); b.set_manifold(True, 0.1); b.load_state_dict(sd)
    c = SnakeVecEnv(num_envs=n, device=0); c.set_manifold(True, 0.1); c.load_state_dict(sd)
    c.set_manifold_cache(torch.zeros((n, STRIDE)))            # control: the same continuation without the caches
    differs = False
    for t in range(3, 6):
        oa, ra, da, _ = a.step(acts[t]); ob, rb, db, _ = b.step(acts[t]); oc, rc, dc, _ = c.step(acts[t])
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db) and torch.equal(a.last_ticks, b.last_ticks)
        assert torch.equal(a.get_manifold_cache(), b.get_manifold_cache())
        differs |= not (torch.equal(oa, oc) and torch.equal(ra, rc))
    assert differs
    off = SnakeVecEnv(num_envs=n, device=0)
    with pytest.raises(ValueError, match="contact model"):
        off.load_state_dict(sd)                               # manifold checkpoint into the default contact model
    with pytest.raises(ValueError, match="contact model"):
        b.load_state_dict(off.state_dict())                   # and the other way round
    other = SnakeVecEnv(num_envs=n, device=0); other.set_manifold(True, 0.0)
    with pytest.raises(ValueError, match="contact model"):
        other.load_state_dict(sd)                             # another warm-start factor
    assert "manifold_cache" not in off.state_dict() and set(off.state_dict()) == {"state", "num_envs", "params"}
    for e in (a, b, c, off, other):
        e.close()


@pytest.mark.gpu
def test_masked_hard_reset_clears_only_the_masked_caches(torch):
    n = 1024
    acts = actions(torch, 5, n, 17)
    a = manifold_env(n)
    for t in range(3):
        a.step(acts[t])
    before = a.get_manifold_cache().clone()
    m = np.random.default_rng(4).random(n) < 0.3
    a.reset(hard=True, mask=m)
    after = a.get_manifold_cache()
    mt = torch.from_numpy(m).cuda()
    assert bool((before[mt] != 0).any())                     # there was something to clear
    assert bool((after[mt] == 0).all()) and torch.equal(after[~mt], before[~mt])
    fresh = SnakeVecEnv(num_envs=n, device=0); fresh.set_manifold(True, 0.1); fresh.reset(hard=True)
    for t in range(3, 5):
        oa, ra, da, _ = a.step(acts[t]); of, rf, df, _ = fresh.step(acts[t])
        assert torch.equal(oa[mt], of[mt]) and torch.equal(ra[mt], rf[mt]) and torch.equal(da[mt], df[mt])
        assert torch.equal(a.last_ticks[mt], fresh.last_ticks[mt])
        assert torch.equal(a.get_manifold_cache()[mt], fresh.get_manifold_cache()[mt])
    a.close(); fresh.close()


@pytest.mark.gpu
def test_set_manifold_cache_refuses_bad_counts(torch):
    n = 64
    acts = actions(torch, 2, n, 19)
    env = manifold_env(n)
    for t in range(2):
        env.step(acts[t])
    before = env.get_manifold_cache().clone()
    assert bool((before[:, COUNTS:] > 0).any())
    for bad in (5.0, 1.5, -1.0, float("nan")):
        c = before.clone(); c[7, COUNTS + 3] = bad
        with pytest.raises(RuntimeError, match="point count"):
            env.set_manifold_cache(c)
        assert torch.equal(env.get_manifold_cache(), before)
    env.set_manifold_cache(before.flip(0))                    # a valid cache goes in
    assert torch.equal(env.get_manifold_cache(), before.flip(0))
    off = SnakeVecEnv(num_envs=n, device=0)
    buf = torch.zeros((n, STRIDE), device="cuda")
    mask = torch.ones(n, dtype=torch.uint8, device="cuda")
    assert off._lib.snk_get_manifold_cache(off._h, buf.data_ptr(), None) == -1
    assert off._lib.snk_set_manifold_cache(off._h, buf.data_ptr(), None) == -1
    assert off._lib.snk_clear_manifold(off._h, mask.data_ptr(), None) == -1
    assert b"manifolds are off" in off._lib.snk_last_error()
    env.close(); off.close()


@pytest.mark.gpu
def test_closing_a_manifold_batch_releases_its_memory(torch):
    """snk_destroy frees the caches (4 224 B per environment) and the row tables (388 MB per device)."""
    import gc

    def round_trip():
        env = manifold_env(65536)
        env.step(torch.zeros((65536, 8), device="cuda"))
        env.close()
        del env
        gc.collect()
        torch.cuda.synchronize(); torch.cuda.empty_cache()

    round_trip()                                              # module loading and torch's first allocations
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(4):
        round_trip()
        free = torch.cuda.mem_get_info()[0]
        assert free >= free0 - (64 << 20), (free0 - free) / 2**20


def test_manifold_cache_entry_points_refuse_a_null_handle():
    import __graft_entry__ as ge
    ge.build()
    from bullet_envs_b200 import _abi
    lib = _abi.load_library()
    assert lib.snk_get_manifold_cache(None, None, None) < 0
    assert lib.snk_set_manifold_cache(None, None, None) < 0
    assert lib.snk_clear_manifold(None, None, None) < 0 and b"null" in lib.snk_last_error()


def test_manifold_trace_and_rollout_kernels_stream_rows_with_async_copies():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    import __graft_entry__ as ge
    ge.build()
    txt = subprocess.run([exe, "-sass", os.path.join(ROOT, "bullet_envs_b200", "csrc", "libsnake_b200.so")], stdout=subprocess.PIPE,
                         text=True, check=True).stdout
    for name in ("_Z25snk_man_step_trace_kernelILb1EE", "_Z22snk_man_rollout_kernelILb1EE"):
        k = [p for p in txt.split("Function : ") if p.startswith(name)]
        assert len(k) == 1, name
        assert k[0].count("LDGSTS") >= 12 and "LDTM" not in k[0] and "STTM" not in k[0], name
