"""Size-independent properties of the CUDA path at BASELINE.json's sizes (no oracle needed): determinism,
independence of an environment from its position in the batch / from the lane and warp that happens to
process it, shard invariance, invariants of the outputs."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU fallback)")
    return torch


def rollout(torch, n, steps, acts, perm=None):
    from bullet_envs_b200 import SnakeVecEnv
    env = SnakeVecEnv(num_envs=n, device=0)
    env.reset(as_torch=True)
    out = []
    for t in range(steps):
        a = acts[t] if perm is None else acts[t][perm]
        obs, rew, done, _ = env.step(a)
        out.append((obs.clone(), rew.clone(), done.clone(), env.last_ticks.clone()))
    st = env.get_state().clone()
    c = env.counters()
    env.close()
    return out, st, c


def test_config2_full_size_determinism_and_invariants(torch):
    """config 2: 4096 environments, 100 env-steps of seeded U[-1,1] actions.  Environments are handed to lanes
    through an atomic counter, so two runs process a given environment on different lanes / warps / row
    storage: bit-identical results show that none of that leaks into the arithmetic."""
    n, steps = 4096, 100
    g = torch.Generator().manual_seed(0)
    acts = (torch.rand((steps, n, 8), generator=g) * 2 - 1).cuda()
    r1, s1, c1 = rollout(torch, n, steps, acts)
    r2, s2, c2 = rollout(torch, n, steps, acts)
    for (o1, w1, d1, t1), (o2, w2, d2, t2) in zip(r1, r2):
        assert torch.equal(o1, o2) and torch.equal(w1, w2) and torch.equal(d1, d2) and torch.equal(t1, t2)
    assert torch.equal(s1, s2)
    ticks = torch.stack([x[3] for x in r1]).float()
    obs = torch.stack([x[0] for x in r1]); rew = torch.stack([x[1] for x in r1]); done = torch.stack([x[2] for x in r1])
    assert torch.isfinite(obs).all() and torch.isfinite(rew).all()
    assert int(ticks.max()) <= 41 and 25 < float(ticks[1:].mean()) < 33          # snake.py:303 cap; ~0.9^k error decay
    assert (obs[..., 51:55].norm(dim=-1) - 1).abs().max() < 1e-5                    # unit base quaternion
    assert (obs[..., :16].abs() <= np.pi / 6 + 0.06).all()                          # joints stay within target range + tolerance
    assert (obs[..., 0:16:2].abs() < 1e-6).all()                                    # gaitSelection 1 never drives the even joints
    post = obs[done]                                                                # done -> post-reset observation
    assert post.shape[0] > 0 and (post[:, :32] == 0).all() and (post[:, 48:51] == 0).all() and (post[:, 54] == 1).all()
    assert c1["nonfinite"] == 0


def test_environment_results_do_not_depend_on_batch_position(torch):
    n, steps = 2048, 6
    g = torch.Generator().manual_seed(3)
    acts = (torch.rand((steps, n, 8), generator=g) * 2 - 1).cuda()
    perm = torch.randperm(n, generator=g).cuda()
    r1, s1, _ = rollout(torch, n, steps, acts)
    r2, s2, _ = rollout(torch, n, steps, acts, perm)
    for (o1, w1, d1, t1), (o2, w2, d2, t2) in zip(r1, r2):
        assert torch.equal(o1[perm], o2) and torch.equal(w1[perm], w2) and torch.equal(d1[perm], d2) and torch.equal(t1[perm], t2)


def test_shards_equal_the_unsharded_batch(torch):
    """one process per GPU shards by contiguous index range: a shard's results are those of the same
    environments inside the full batch (W = 1 vs W = 2 bit-identical)."""
    from bullet_envs_b200.dist import shard_range
    n, steps = 1000, 5
    g = torch.Generator().manual_seed(5)
    acts = (torch.rand((steps, n, 8), generator=g) * 2 - 1).cuda()
    full, _, _ = rollout(torch, n, steps, acts)
    for rank in range(2):
        lo, hi = shard_range(n, rank, 2)
        part, _, _ = rollout(torch, hi - lo, steps, acts[:, lo:hi].contiguous())
        for (o1, w1, d1, t1), (o2, w2, d2, t2) in zip(full, part):
            assert torch.equal(o1[lo:hi], o2) and torch.equal(w1[lo:hi], w2) and torch.equal(d1[lo:hi], d2)


def test_warp_count_and_hand_out_policy_do_not_change_results(torch):
    """The number of working warps per SM and the hand-out policy (warp-major first wave, longest-first order) may not change a bit
    of the results.  70 000 environments (about two waves of the grid), forced to 6 / 7 / 4 warps and to the CTA-major and fully
    dynamic hand-outs and the index order, in subprocesses; checksums."""
    import os, subprocess, sys
    code = ("import torch, hashlib; from bullet_envs_b200 import SnakeVecEnv;"
            "g=torch.Generator().manual_seed(4); a=(torch.rand((2,70000,8),generator=g)*2-1).cuda();"
            "e=SnakeVecEnv(num_envs=70000,device=0); e.reset(as_torch=True);"
            "h=hashlib.sha256();\n"
            "for t in range(2):\n"
            "    o,r,d,_=e.step(a[t]); h.update(o.cpu().numpy().tobytes()); h.update(r.cpu().numpy().tobytes()); h.update(e.last_ticks.cpu().numpy().tobytes())\n"
            "print('SUM', h.hexdigest())")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sums = []
    for extra in ({}, {"SNK_EXACT_WARPS": "6"}, {"SNK_EXACT_WARPS": "7"}, {"SNK_EXACT_WARPS": "4"}, {"SNK_EXACT_SPREAD": "0"}, {"SNK_EXACT_SPREAD": "2"},
                  {"SNK_EXACT_ORDER": "index"}, {"SNK_EXACT_BALANCE": "0"}):
        env = dict(os.environ, PYTHONPATH=root, **extra)
        out = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
        assert out.returncode == 0, out.stderr[-2000:]
        sums.append([l for l in out.stdout.splitlines() if l.startswith("SUM")][0])
    assert len(set(sums)) == 1, sums


def test_split_hand_out_does_not_change_results(torch):
    """Split hand-out (SplitCta in csrc/snake_exact.cu): with n = k L + r environments and r <= L / 2 the r shortest env-steps are run in
    two parts by two lanes of a CTA (parked at a tick boundary, finished when the whole env-steps have run out).  Not a bit of the
    results may depend on it: 50 000 and 131 072 environments (1.3 and 3.46 waves of the 37 888-lane grid), three env-steps, the third
    with repeated actions for a quarter of the batch (zero-tick env-steps, which end inside their first part), split on / off, first
    parts of 30 % and 90 % of the predicted ticks, and the two pools off as well; checksums of observations, rewards, dones, ticks and
    the state array, in subprocesses (the switches are read at snk_create)."""
    import os, subprocess, sys
    code = ("import sys, torch, hashlib; from bullet_envs_b200 import SnakeVecEnv;"
            "n=int(sys.argv[1]); g=torch.Generator().manual_seed(21); a=(torch.rand((3,n,8),generator=g)*2.4-1.2); a[2,::4]=a[1,::4]; a=a.cuda();"
            "e=SnakeVecEnv(num_envs=n,device=0); e.reset(as_torch=True);"
            "h=hashlib.sha256(); dn=0\n"
            "for t in range(3):\n"
            "    o,r,d,_=e.step(a[t]); dn+=int(d.sum())\n"
            "    for x in (o,r,d,e.last_ticks,e.get_state()): h.update(x.cpu().numpy().tobytes())\n"
            "print('SUM', h.hexdigest(), dn, e.counters()['ticks'])")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for n in (50000, 131072):
        sums = []
        for extra in ({}, {"SNK_EXACT_SPLIT": "0"}, {"SNK_EXACT_SPLIT_FRAC": "30"}, {"SNK_EXACT_SPLIT_FRAC": "90"}, {"SNK_EXACT_SPLIT": "0", "SNK_EXACT_BALANCE": "0"}):
            env = dict(os.environ, PYTHONPATH=root, **extra)
            out = subprocess.run([sys.executable, "-c", code, str(n)], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
            assert out.returncode == 0, out.stderr[-2000:]
            sums.append([l for l in out.stdout.splitlines() if l.startswith("SUM")][0])
        assert len(set(sums)) == 1, sums


def test_split_hand_out_stress(torch):
    """No sanitizer on this pool: the park / claim / resume protocol of the split hand-out (CTA-scope fence + flag word, per-CTA claim
    counter) is exercised instead -- 40 consecutive env-steps (episodes end and restart on the way) at three batch sizes (r / L = 0.19,
    0.85 and 0.46 of a wave left over), every step a fresh launch with fresh parked env-steps, against the same run without splitting."""
    import os, subprocess, sys
    code = ("import sys, torch, hashlib; from bullet_envs_b200 import SnakeVecEnv;"
            "n=int(sys.argv[1]); g=torch.Generator(device='cuda').manual_seed(33);"
            "e=SnakeVecEnv(num_envs=n,device=0); e.reset(as_torch=True);"
            "h=hashlib.sha256(); dn=0\n"
            "for t in range(40):\n"
            "    a=torch.rand((n,8),generator=g,device='cuda')*2.6-1.3\n"
            "    if t % 5 == 4: a[::3]=prev[::3]\n"
            "    prev=a; o,r,d,_=e.step(a); dn+=int(d.sum())\n"
            "    for x in (o,r,d,e.last_ticks): h.update(x.cpu().numpy().tobytes())\n"
            "h.update(e.get_state().cpu().numpy().tobytes()); print('SUM', h.hexdigest(), dn)")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for n in (45000, 70000, 131072):
        sums = []
        for extra in ({}, {"SNK_EXACT_SPLIT": "0"}):
            env = dict(os.environ, PYTHONPATH=root, **extra)
            out = subprocess.run([sys.executable, "-c", code, str(n)], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
            assert out.returncode == 0, out.stderr[-2000:]
            sums.append([l for l in out.stdout.splitlines() if l.startswith("SUM")][0])
        assert len(set(sums)) == 1, sums
        assert int(sums[0].split()[2]) > 0      # episodes did end on the way


def test_checkpoint_resume_is_bit_exact(torch):
    from bullet_envs_b200 import SnakeVecEnv
    n = 300
    g = torch.Generator().manual_seed(11)
    acts = (torch.rand((6, n, 8), generator=g) * 2 - 1).cuda()
    a = SnakeVecEnv(num_envs=n, device=0); a.reset(as_torch=True)
    for t in range(3):
        a.step(acts[t])
    sd = a.state_dict()
    b = SnakeVecEnv(num_envs=n, device=0); b.load_state_dict(sd)
    for t in range(3, 6):
        oa, ra, da, _ = a.step(acts[t]); ob, rb, db, _ = b.step(acts[t])
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)
    with pytest.raises(ValueError):
        SnakeVecEnv(num_envs=n + 1, device=0).load_state_dict(sd)
    a.close(); b.close()
