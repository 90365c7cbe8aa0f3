"""GPU: the PPO rollout kernels (include/ppo_b200.h) against plain PyTorch fp32 /
numpy restatements of the stable-baselines3 operations they replace.

Tolerances: the policy forward computes in bf16 x bf16 -> fp32 with bf16
activations and tanh.approx; against an fp32 PyTorch forward of the same
(bf16-rounded) weights the action mean / value must agree to 3e-2 absolute
(pre-activations are O(1)); everything else (sampling algebra, GAE, running
statistics, reward normalisation) is fp32/fp64 arithmetic compared at 1e-5.
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    import __graft_entry__ as ge

    ge.build()
    import fpv_drone_rl_agent_b200 as pkg
    from fpv_drone_rl_agent_b200 import _lib, ppo

    return pkg, _lib, ppo


def test_tcgen05_gemm_hook(env):
    pkg, _lib, ppo = env
    L = _lib.lib()
    torch.manual_seed(0)
    for n, k in [(16, 16), (128, 128), (256, 32), (16, 256), (64, 96)]:
        A = torch.randn(128, k, device="cuda").to(torch.bfloat16)
        B = torch.randn(n, k, device="cuda").to(torch.bfloat16)
        D = torch.zeros(128, n, device="cuda")
        assert L.ppo_test_gemm(A.data_ptr(), B.data_ptr(), D.data_ptr(), n, k, None) == 0
        torch.cuda.synchronize()
        ref = A.float() @ B.float().t()
        assert (D - ref).abs().max().item() < 1e-3 * max(1.0, ref.abs().max().item())


def _model(ppo, seed=0):
    torch.manual_seed(seed)
    m = ppo.ActorCritic().cuda()
    with torch.no_grad():  # make the heads non-trivial (SB3 init has gain 0.01 on the action head)
        m.mu.weight.mul_(30.0)
        m.mu.bias.uniform_(-0.2, 0.2)
        m.v.bias.fill_(0.3)
        m.log_std.copy_(torch.tensor([-0.5, 0.0, 0.3, -1.0]))
        for lin in (m.pi1, m.pi2, m.vf1, m.vf2):
            lin.bias.uniform_(-0.3, 0.3)
    return m


def _bf16_weights(m):
    """fp32 model whose weights are the bf16-rounded ones the kernel uses."""
    import copy

    r = copy.deepcopy(m)
    with torch.no_grad():
        for lin in (r.pi1, r.pi2, r.mu, r.vf1, r.vf2, r.v):
            lin.weight.copy_(lin.weight.to(torch.bfloat16).float())
    return r


@pytest.mark.parametrize("n", [1, 100, 128, 4096, 50_000])
def test_policy_forward_matches_torch(env, n):
    pkg, _lib, ppo = env
    m = _model(ppo)
    pol = ppo.PackedPolicy(m, "cuda")
    torch.manual_seed(1)
    obs = torch.randn(n, 20, device="cuda") * 2.0
    st = ppo.RunningStats(20, "cuda")
    st.mean.copy_(torch.randn(20, device="cuda") * 0.3)
    st.inv_std.copy_(torch.rand(20, device="cuda") + 0.5)
    acts = torch.zeros(n, 4, device="cuda"); eacts = torch.zeros(n, 4, device="cuda")
    vals = torch.zeros(n, device="cuda"); logp = torch.zeros(n, device="cuda"); on = torch.zeros(n, 20, device="cuda")
    ppo.policy_forward(pol, obs, obs_stats=st, obs_clip=3.0, seed=5, row0=7, step=11, actions=acts, env_actions=eacts, values=vals,
                       log_probs=logp, obs_norm=on)
    torch.cuda.synchronize()
    xn = torch.clamp((obs - st.mean) * st.inv_std, -3.0, 3.0)
    assert (on - xn).abs().max().item() < 1e-5
    with torch.no_grad():
        mean_ref, v_ref = _bf16_weights(m)(xn.to(torch.bfloat16).float())
    std = m.log_std.exp()
    z = (acts - mean_ref) / std  # implied standard normal draws
    # value / mean accuracy through the implied noise is checked with the deterministic pass below
    d_acts = torch.zeros(n, 4, device="cuda"); d_vals = torch.zeros(n, device="cuda")
    ppo.policy_forward(pol, obs, obs_stats=st, obs_clip=3.0, deterministic=True, actions=d_acts, values=d_vals)
    torch.cuda.synchronize()
    assert (d_acts - mean_ref).abs().max().item() < 3e-2, (d_acts - mean_ref).abs().max().item()
    assert (d_vals - v_ref).abs().max().item() < 3e-2
    assert (vals - d_vals).abs().max().item() == 0.0
    # sampling algebra: a = mean + std * z, logp = sum(-z^2/2 - log_std - ln sqrt(2 pi)), env action = clip(a)
    z_k = (acts - d_acts) / std
    lp = (-0.5 * z_k * z_k - m.log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
    assert (lp - logp).abs().max().item() < 2e-3
    assert torch.equal(eacts, acts.clamp(-1, 1))
    if n >= 4096:
        assert abs(z_k.mean().item()) < 0.02 and abs(z_k.std().item() - 1.0) < 0.02
        assert abs(torch.corrcoef(z_k.t())[0, 1].item()) < 0.05
    # determinism and counter semantics
    a2 = torch.zeros_like(acts)
    ppo.policy_forward(pol, obs, obs_stats=st, obs_clip=3.0, seed=5, row0=7, step=11, actions=a2)
    a3 = torch.zeros_like(acts)
    base = torch.tensor([4], dtype=torch.int64, device="cuda")
    ppo.policy_forward(pol, obs, obs_stats=st, obs_clip=3.0, seed=5, row0=7, step=7, step_base=base, actions=a3)
    a4 = torch.zeros_like(acts)
    ppo.policy_forward(pol, obs, obs_stats=st, obs_clip=3.0, seed=5, row0=7, step=12, actions=a4)
    torch.cuda.synchronize()
    assert torch.equal(a2, acts) and torch.equal(a3, acts) and not torch.equal(a4, acts)
    if n > 200:  # sharding invariance: rows 100.. of the batch == a separate call with row0 shifted
        a5 = torch.zeros(n - 100, 4, device="cuda")
        ppo.policy_forward(pol, obs[100:], obs_stats=st, obs_clip=3.0, seed=5, row0=107, step=11, actions=a5)
        torch.cuda.synchronize()
        assert torch.equal(a5, acts[100:])


@pytest.mark.parametrize("T,n", [(37, 1000), (8, 4096), (128, 4096), (2048, 33), (33, 31), (64, 200_000), (5, 300_000)])
def test_gae_matches_sb3_recurrence(env, T, n):
    """Both GAE kernels (warp scan over time for small batches, one thread per env for large ones) against the SB3 loop."""
    pkg, _lib, ppo = env
    g = torch.Generator(device="cuda").manual_seed(0)
    rew = torch.randn(T, n, device="cuda", generator=g)
    val = torch.randn(T, n, device="cuda", generator=g)
    done = (torch.rand(T, n, device="cuda", generator=g) < 0.05).to(torch.uint8)
    last = torch.randn(n, device="cuda", generator=g)
    adv = torch.zeros(T, n, device="cuda"); ret = torch.zeros(T, n, device="cuda")
    ppo.gae(rew, val, done, last, 0.99, 0.95, adv, ret)
    torch.cuda.synchronize()
    r, v, d, lv = rew.double().cpu().numpy(), val.double().cpu().numpy(), done.cpu().numpy().astype(np.float64), last.double().cpu().numpy()
    a = np.zeros((T, n)); gae = np.zeros(n)
    for t in reversed(range(T)):  # SB3 RolloutBuffer.compute_returns_and_advantage
        nv = lv if t == T - 1 else v[t + 1]
        nnt = 1.0 - d[t]
        delta = r[t] + 0.99 * nv * nnt - v[t]
        gae = delta + 0.99 * 0.95 * nnt * gae
        a[t] = gae
    np.testing.assert_allclose(adv.cpu().numpy(), a, rtol=0, atol=2e-4)
    np.testing.assert_allclose(ret.cpu().numpy(), a + v, rtol=0, atol=2e-4)


def test_running_stats_and_reward_normalisation(env):
    pkg, _lib, ppo = env
    L = _lib.lib()
    n, dim = 5000, 20
    st = ppo.RunningStats(dim, "cuda")
    mean, var, count = np.zeros(dim), np.ones(dim), 1e-4
    rng = np.random.default_rng(0)
    for it in range(4):
        x = (rng.normal(size=(n, dim)) * (1 + it) + it).astype(np.float32)
        st.update(torch.from_numpy(x).cuda())
        bm, bv, bc = x.astype(np.float64).mean(0), x.astype(np.float64).var(0), n  # VecNormalize RunningMeanStd.update
        delta, tot = bm - mean, count + bc
        m2 = var * count + bv * bc + delta**2 * count * bc / tot
        mean, var, count = mean + delta * bc / tot, m2 / tot, tot
    torch.cuda.synchronize()
    s = st.stats.cpu().numpy()
    np.testing.assert_allclose(s[:dim], mean, rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(s[dim:2 * dim], var, rtol=1e-7)
    assert abs(s[2 * dim] - count) < 1e-6
    np.testing.assert_allclose(st.inv_std.cpu().numpy(), 1 / np.sqrt(var + 1e-8), rtol=1e-5)
    # reward path of VecNormalize.step_wait
    rs = ppo.RunningStats(1, "cuda")
    acc = torch.zeros(n, device="cuda")
    ret, rmean, rvar, rcount = np.zeros(n), 0.0, 1.0, 1e-4
    for it in range(5):
        r = rng.normal(size=n).astype(np.float32) * 3
        te = (rng.random(n) < 0.1).astype(np.uint8); tr = (rng.random(n) < 0.05).astype(np.uint8)
        out = torch.zeros(n, device="cuda"); dn = torch.zeros(n, dtype=torch.uint8, device="cuda")
        assert L.ppo_reward_normalize(torch.from_numpy(r).cuda().data_ptr(), torch.from_numpy(te).cuda().data_ptr(), torch.from_numpy(tr).cuda().data_ptr(),
                                      acc.data_ptr(), n, 0.99, 10.0, 1e-8, rs.stats.data_ptr(), out.data_ptr(), dn.data_ptr(), rs.scratch.data_ptr(), None) == 0
        torch.cuda.synchronize()
        ret = ret * 0.99 + r
        bm, bv = ret.mean(), ret.var()
        delta, tot = bm - rmean, rcount + n
        m2 = rvar * rcount + bv * n + delta**2 * rcount * n / tot
        rmean, rvar, rcount = rmean + delta * n / tot, m2 / tot, tot
        exp = np.clip(r / np.sqrt(rvar + 1e-8), -10, 10)
        ret[(te | tr) > 0] = 0.0
        np.testing.assert_allclose(out.cpu().numpy(), exp, rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose(acc.cpu().numpy(), ret, rtol=1e-5, atol=1e-5)
        assert np.array_equal(dn.cpu().numpy(), te | tr)


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("n", [1000, 131072, 200_001])
def test_fused_statistics_forward_equals_the_two_launches(env, n, fused):
    """ppo_policy_forward_stats (VecNormalize's obs_rms.update + normalize_obs + the policy forward in one launch) against
    ppo_running_stats_update followed by ppo_policy_forward: the running statistics agree to fp64 rounding (the per-CTA partial
    sums are grouped differently), the fp32 (mean, inv_std) to one ulp, and the outputs to what one ulp of the normalisation
    moves them.  Three successive batches through the same buffers check that the in-kernel ticket / flag words re-arm."""
    pkg, _lib, ppo = env
    m = _model(ppo, seed=3)
    pol = ppo.PackedPolicy(m, "cuda:0")
    a_stats, b_stats = ppo.RunningStats(20, "cuda:0"), ppo.RunningStats(20, "cuda:0")
    g = torch.Generator(device="cuda").manual_seed(n)
    for rep in range(3):
        x = torch.randn(n, 20, device="cuda", generator=g) * (1.0 + rep) + torch.linspace(-2, 2, 20, device="cuda")
        out_a = [torch.zeros(n, 4, device="cuda"), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda"), torch.zeros(n, 20, device="cuda")]
        out_b = [torch.zeros_like(t) for t in out_a]
        a_stats.update(x)
        ppo.policy_forward(pol, x, obs_stats=a_stats, obs_clip=10.0, seed=5, step=rep, actions=out_a[0], values=out_a[1], log_probs=out_a[2], obs_norm=out_a[3])
        ppo.policy_forward(pol, x, obs_stats=b_stats, obs_clip=10.0, seed=5, step=rep, actions=out_b[0], values=out_b[1], log_probs=out_b[2], obs_norm=out_b[3],
                           update_stats=True, fused_stats=fused)  # fused: one launch; not fused: two launches chained as programmatic dependents
        torch.cuda.synchronize()
        assert torch.allclose(a_stats.stats, b_stats.stats, rtol=1e-12, atol=1e-12), (a_stats.stats - b_stats.stats).abs().max()
        assert float(b_stats.stats[40]) == pytest.approx(1e-4 + (rep + 1) * n)
        assert torch.allclose(a_stats.mean, b_stats.mean, rtol=3e-7, atol=1e-7) and torch.allclose(a_stats.inv_std, b_stats.inv_std, rtol=3e-7)
        assert (out_a[3] - out_b[3]).abs().max().item() < 1e-5
        assert (out_a[1] - out_b[1]).abs().max().item() < 2e-2 and (out_a[0] - out_b[0]).abs().max().item() < 2e-2  # bf16 staging of a 1-ulp-different input
        assert (out_a[1] - out_b[1]).abs().mean().item() < 1e-4
    # numpy restatement of the merged moments
    assert torch.isfinite(b_stats.stats).all()


def test_time_limit_bootstrap(env):
    """Envs that hover into the 402-step limit get reward += gamma * V(terminal_obs) (SB3 collect_rollouts)."""
    pkg, _lib, ppo = env
    thr = float(np.sqrt(0.1 * 9.81 / 4.0))
    n = 300
    cfg = pkg.default_config()
    cfg.update(start_pos=[0, 0, 2.8], spawn_throttle=thr, reset_idle_steps=0, noise=0, max_steps=5)  # 0.2 m below the dome
    sim = pkg.QuadXSim(n, cfg, seed=0)
    m = _model(ppo)
    pol = ppo.PackedPolicy(m, "cuda")
    obs = torch.zeros(n, 20, device="cuda"); rew = torch.zeros(n, device="cuda"); tobs = torch.zeros(n, 20, device="cuda")
    te = torch.zeros(n, dtype=torch.uint8, device="cuda"); tr = torch.zeros(n, dtype=torch.uint8, device="cuda")
    sim.reset(obs)
    a = torch.zeros(n, 4, device="cuda"); a[:, 3] = 2 * thr - 1
    a[::3, 3] = 1.0  # every third env rockets out of the dome instead (terminated, not truncated)
    queue = sim.done_queue()
    seen_trunc = seen_term = 0
    for k in range(12):
        sim.step_begin(a, obs, rew, te, tr, tobs)
        before = rew.clone()
        ppo.bootstrap_truncated(pol, tobs, None, 0.0, queue, te, tr, 0.99, rew)
        sim.step_end(obs)
        torch.cuda.synchronize()
        trunc_only = tr.bool() & ~te.bool()
        with torch.no_grad():
            _, v = _bf16_weights(m)(tobs.to(torch.bfloat16).float())
        exp = before + 0.99 * v * trunc_only
        assert (rew - exp)[trunc_only].abs().max().item() < 3e-2 if trunc_only.any() else True
        assert torch.equal(rew[~trunc_only], before[~trunc_only])
        # the other order (ppo_bootstrap_truncated_first + ppo_reward_normalize_add) gives the same rewards as
        # ppo_reward_normalize + ppo_bootstrap_truncated, up to the one rounding of fma(gamma, V, r) vs gamma V + r
        outs = []
        for first in (False, True):
            st, acc = ppo.RunningStats(1, "cuda"), torch.zeros(n, device="cuda")
            st.stats[1] = 4.0  # a return variance that is not 1
            out, dn = torch.full((n,), 123.0, device="cuda"), torch.zeros(n, dtype=torch.uint8, device="cuda")
            boot = (pol, tobs, None, 0.0, queue, te, tr, 0.99, out)
            nrm = (before, te, tr, acc, st, 0.99, 10.0, out, dn)
            if first:
                ppo.bootstrap_truncated(*boot, first=True)
                ppo.reward_normalize(*nrm, add=True)
            else:
                ppo.reward_normalize(*nrm)
                ppo.bootstrap_truncated(*boot)
            torch.cuda.synchronize()
            outs.append((out.clone(), dn.clone(), acc.clone(), st.stats.clone()))
        assert (outs[0][0] - outs[1][0]).abs().max().item() < 1e-5 and torch.equal(outs[0][1], outs[1][1])
        assert torch.equal(outs[0][2], outs[1][2]) and torch.equal(outs[0][3], outs[1][3])
        seen_trunc += int(trunc_only.sum()); seen_term += int(te.sum())
    assert seen_trunc > 0 and seen_term > 0


def test_rollout_graph_equals_eager_and_training_improves(env):
    pkg, _lib, ppo = env
    cfgs = [ppo.PPOConfig(n_envs=2048, n_steps=16, seed=3, use_cuda_graph=g, n_epochs=2, batch_size=8192) for g in (False, True)]
    trainers = [ppo.PPOTrainer(c, device="cuda") for c in cfgs]
    for it in range(2):
        for t in trainers:
            t.rollout.collect()
        torch.cuda.synchronize()
        a, b = trainers[0].rollout, trainers[1].rollout
        for name in ("obs", "actions", "log_probs", "values", "rewards", "dones", "advantages", "returns"):
            assert torch.equal(getattr(a, name), getattr(b, name)), name
    # SB3 semantics of the buffers
    ro = trainers[1].rollout
    assert ro.obs.abs().max().item() <= 10.0 + 1e-6 and ro.rewards.abs().max().item() <= 10.0 + 1e-6
    assert torch.isfinite(ro.advantages).all() and torch.isfinite(ro.returns).all()
    assert torch.allclose(ro.returns - ro.advantages, ro.values, atol=1e-5)
    # a few PPO iterations run end to end and produce finite statistics
    t = trainers[1]
    out = None
    for it in range(3):
        out = t.learn_iteration()
    assert all(math.isfinite(out[k]) for k in ("pg", "vf", "kl")) and out["timesteps"] == 3 * 2048 * 16


def test_yaw_rollout_on_device(env):
    """BASELINE configs[2]: the yaw task with the full on-device PPO rollout (12-D obs, 1-D action)."""
    pkg, _lib, ppo = env
    cfg = ppo.PPOConfig(n_envs=4096, n_steps=16, seed=1, n_epochs=1, batch_size=16384, log_std_init=-1.0)
    t = ppo.PPOTrainer(cfg, device="cuda", task=pkg.QX_TASK_YAW)
    ro = t.rollout
    assert ro.obs.shape == (16, 4096, 12) and ro.actions.shape == (16, 4096, 1)
    out = t.learn_iteration()
    assert math.isfinite(out["pg"]) and math.isfinite(out["vf"])
    assert torch.isfinite(ro.advantages).all() and ro.obs.abs().max().item() <= 10.0 + 1e-6
    # the stored log-probs are those of the stored actions under the stored (normalised) observations
    with torch.no_grad():
        ro.collect()
        torch.cuda.synchronize()
        v, lp, _ = t.model.evaluate_actions(ro.obs.view(-1, 12), ro.actions.view(-1, 1))
    assert (lp - ro.log_probs.view(-1)).abs().max().item() < 0.2 and (v - ro.values.view(-1)).abs().max().item() < 5e-2
