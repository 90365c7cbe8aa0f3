"""GPU: the SAC actor kernel (sac::actor_forward_kernel, K8, sac_actor_forward) row by row against a float64 reference that
rounds where the kernel rounds, in a CUDA graph, inside ppo.evaluate_policy, and PPO archives through sac.load_sb3_zip.

The reference (``_reference``) follows the kernel's rounding points:
  x_hat = clamp((x - mean) * inv_std, +-clip)      fp32, two roundings: obs_norm_out must equal it bit for bit
  X = bf16_rne(x_hat)
  p1 = fp32(fp32(X . W1^T) + b1);  h1 = bf16_rne(relu(p1))      products of bf16 values are exact in fp64
  p2, h2 the same for layer 2;  m = fp32(fp32(h2 . Wmu^T) + b_mu);  a = fp32(tanh(m))
What it cannot know is the order and rounding of the tensor core's fp32 accumulation.  So for every row and unit it carries a
rigorous bound on |accumulator - exact sum| (GAMMA x K x the sum of |terms|, plus what the input's own interval contributes),
maps the two ends of that interval through the same monotone roundings (fp32 bias add, ReLU, bf16 / tanh, fp32), and
requires every action of every row to lie inside the resulting interval.  Where an interval spans a bf16 rounding boundary
the kernel may take either side; elsewhere the interval is a single value and the check is exact.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# name -> (obs_dim, act_dim, net_arch)
SHAPES = {"hover128": (20, 4, (128, 128)), "hover64": (20, 4, (64, 64)), "yaw128": (12, 1, (128, 128)), "yaw64": (12, 1, (64, 64))}
ROW_COUNTS = [1, 127, 128, 129, 4096, 131_072]
GAMMA = 2.0 ** -22  # per accumulated term: twice the fp32 unit roundoff, for an accumulation order and rounding we do not know


@pytest.fixture(scope="module")
def env():
    import __graft_entry__ as ge

    ge.build()
    from fpv_drone_rl_agent_b200 import _lib, ppo, sac

    return _lib, ppo, sac


def _actor(sac, shape, seed=0):
    """An SB3-initialised actor with a strong action head (so the squash saturates on some rows) and non-zero biases."""
    od, ad, h = SHAPES[shape]
    torch.manual_seed(seed)
    m = sac.SacActor(od, ad, h)
    with torch.no_grad():
        m.mu.weight.mul_(8.0)
        for lin in (m.latent_pi[0], m.latent_pi[2], m.mu):
            lin.bias.uniform_(-0.3, 0.3)
    return m.cuda()


def _obs(n, od, stride, offset, seed):
    """[n, od] raw observations, a view of an [n, stride] buffer starting `offset` floats in (offset 1: not 16-byte aligned)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    buf = torch.randn(n * stride + offset, device="cuda", generator=g) * 2.0
    return buf[offset:].view(n, stride)[:, :od]


def _norm(od, seed):
    g = torch.Generator(device="cuda").manual_seed(1000 + seed)
    return torch.randn(od, device="cuda", generator=g) * 0.3, torch.rand(od, device="cuda", generator=g) + 0.5


def _normalize(obs, mean, inv_std, clip):
    x = obs.float()
    if mean is None:
        return x.clone()
    x = (x - mean) * inv_std
    c = clip if clip > 0 else 3.0e38
    return x.clamp(-c, c)


def _layer(x, dx, w, b, act):
    """one layer over the interval x +- dx (float64): -> (reference value, lower end, upper end) after `act`"""
    exact = x @ w.t()
    err = GAMMA * w.shape[1] * ((x.abs() + dx) @ w.abs().t()) + dx @ w.abs().t()
    ref, lo, hi = (act((e.float() + b).double()) for e in (exact, exact - err, exact + err))
    return ref, lo, hi


def _bf16_relu(p):
    return torch.relu(p).float().to(torch.bfloat16).double()


def _reference(packed, obs, mean=None, inv_std=None, clip=10.0, roll=0):
    """-> (x_hat fp32 [n, od], actions ref / lower / upper fp64 [n, ad]); roll: the reference of the wrong rows (sensitivity)"""
    od, ad = packed.model.obs_dim, packed.model.act_dim
    xh = _normalize(obs, mean, inv_std, clip)
    X = torch.roll(xh, roll, 0).to(torch.bfloat16).double()
    w1, w2, wmu = packed.w1.double()[:, :od], packed.w2.double(), packed.w_mu.double()[:ad]
    zero = torch.zeros_like(X)
    h1, lo1, hi1 = _layer(X, zero, w1, packed.b1, _bf16_relu)
    d1 = torch.maximum(hi1 - h1, h1 - lo1)
    h2, lo2, hi2 = _layer(h1, d1, w2, packed.b2, _bf16_relu)
    d2 = torch.maximum(hi2 - h2, h2 - lo2)
    tanh32 = lambda m: torch.tanh(m).float().double()  # noqa: E731
    a, lo, hi = _layer(h2, d2, wmu, packed.b_mu[:ad], tanh32)
    f = lambda t, d: torch.nextafter(t.float(), torch.full_like(t.float(), d)).double()  # noqa: E731  one fp32 ulp for the fp64 tanh
    return xh, a, f(lo, -2.0), f(hi, 2.0), int(((d1 > 0).any(1) | (d2 > 0).any(1)).sum())


def _check(actions, a_ref, lo, hi):
    """-> number of rows with an action outside its interval"""
    a = actions.double()
    return int(((a < lo) | (a > hi)).any(1).sum())


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("n", ROW_COUNTS)
def test_forward_matches_reference(env, shape, n):
    """Every action of every row inside its interval, obs_norm_out bit for bit.  The row count picks the input layout
    (stride obs_dim, 24 or obs_dim + 1; base 16-byte aligned or one float off: vector and scalar load paths) and the
    normalisation (statistics with clip 3, statistics without clip, none)."""
    _lib, ppo, sac = env
    od, ad, _ = SHAPES[shape]
    k = ROW_COUNTS.index(n) + list(SHAPES).index(shape)
    stride, offset, mode = (od, 24, od + 1)[k % 3], k % 2, (k // 2) % 3
    packed = sac.PackedSacActor(_actor(sac, shape, seed=k), "cuda")
    obs = _obs(n, od, stride, offset, seed=n + k)
    mean, inv = _norm(od, k)
    kw = [dict(mean=mean, inv_std=inv, clip=3.0), dict(mean=mean, inv_std=inv, clip=0.0), dict(mean=None, inv_std=None, clip=3.0)][mode]
    act, on = torch.full((n, ad), 7.0, device="cuda"), torch.full((n, od), 7.0, device="cuda")
    norm = (kw["mean"], kw["inv_std"]) if kw["mean"] is not None else None
    sac.sac_actor_forward(packed, obs, norm=norm, obs_clip=kw["clip"], actions=act, obs_norm=on)
    xh, a_ref, lo, hi, n_wide = _reference(packed, obs, **kw)
    torch.cuda.synchronize()
    assert torch.equal(on, xh), "obs_norm_out is not the fp32 normalisation"
    bad = _check(act, a_ref, lo, hi)
    dev = float((act.double() - a_ref).abs().max())
    width = (hi - lo).amax(1)
    print(f"measured {shape} n={n} stride {stride} offset {offset} mode {mode}: {n_wide} rows with a rounding-ambiguous unit, "
          f"interval width median {float(width.median()):.2e} max {float(width.max()):.2e}, max |a - a_ref| {dev:.3e}, rows outside {bad}")
    assert bad == 0
    with torch.no_grad():  # the torch SacActor (fp32, no bf16) is the same function up to the bf16 roundings
        assert (packed.model(xh) - act).abs().max().item() < 0.1


@pytest.mark.parametrize("shape", ["hover128", "yaw128"])
def test_sensitivity(env, shape):
    """The interval check fails, on most rows, for the reference of the neighbouring row."""
    _lib, ppo, sac = env
    od, ad, _ = SHAPES[shape]
    n = 131_072
    packed = sac.PackedSacActor(_actor(sac, shape, seed=3), "cuda")
    obs = _obs(n, od, od, 0, seed=3)
    mean, inv = _norm(od, 3)
    act = torch.empty(n, ad, device="cuda")
    sac.sac_actor_forward(packed, obs, norm=(mean, inv), obs_clip=3.0, actions=act)
    _, a_ref, lo, hi, _ = _reference(packed, obs, mean, inv, 3.0)
    assert _check(act, a_ref, lo, hi) == 0
    _, a_ref, lo, hi, _ = _reference(packed, obs, mean, inv, 3.0, roll=1)
    assert _check(act, a_ref, lo, hi) > n // 2


@pytest.mark.parametrize("shape", ["hover128", "yaw128"])
def test_misaligned_outputs_and_graph(env, shape):
    """Outputs at a storage offset of one float (scalar stores) and a launch captured in a CUDA graph both give the eager,
    aligned results bit for bit."""
    _lib, ppo, sac = env
    od, ad, _ = SHAPES[shape]
    n = 131_072 + 77
    packed = sac.PackedSacActor(_actor(sac, shape, seed=4), "cuda")
    mean, inv = _norm(od, 4)
    obs = _obs(n, od, 24, 0, seed=4)
    base, base_n = torch.empty(n, ad, device="cuda"), torch.empty(n, od, device="cuda")
    sac.sac_actor_forward(packed, obs, norm=(mean, inv), obs_clip=3.0, actions=base, obs_norm=base_n)
    odd_a = torch.full((n * ad + 1,), 7.0, device="cuda")[1:].view(n, ad)
    odd_n = torch.full((n * od + 1,), 7.0, device="cuda")[1:].view(n, od)
    buf = torch.zeros(n * 24 + 1, device="cuda")
    shifted = buf[1:].view(n, 24)[:, :od]  # the same rows one float off 16-byte alignment
    shifted.copy_(obs)
    sac.sac_actor_forward(packed, shifted, norm=(mean, inv), obs_clip=3.0, actions=odd_a, obs_norm=odd_n)
    g_a, g_n = torch.zeros(n, ad, device="cuda"), torch.zeros(n, od, device="cuda")
    graph = ppo._capture(lambda: sac.sac_actor_forward(packed, obs, norm=(mean, inv), obs_clip=3.0, actions=g_a, obs_norm=g_n), "cuda")
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(odd_a, base) and torch.equal(odd_n, base_n)
    assert torch.equal(g_a, base) and torch.equal(g_n, base_n)


def test_binding_rejects_bad_buffers(env):
    _lib, ppo, sac = env
    n = 256
    packed = sac.PackedSacActor(_actor(sac, "hover128"), "cuda")
    obs = _obs(n, 20, 20, 0, seed=1)
    with pytest.raises(ValueError, match="actions"):
        sac.sac_actor_forward(packed, obs, actions=torch.zeros(n, 8, device="cuda")[:, :4])
    with pytest.raises(ValueError, match="obs_norm"):
        sac.sac_actor_forward(packed, obs, actions=torch.zeros(n, 4, device="cuda"), obs_norm=torch.zeros(n, 21, device="cuda"))
    with pytest.raises(ValueError, match="obs"):
        sac.sac_actor_forward(packed, obs[:, :12], actions=torch.zeros(n, 4, device="cuda"))
    with pytest.raises(ValueError, match="mean"):
        sac.sac_actor_forward(packed, obs, actions=torch.zeros(n, 4, device="cuda"), norm=(torch.zeros(12, device="cuda"), torch.ones(20, device="cuda")))


# ---------------------------------------------------------------------------------------------------------------------------
# evaluation
# ---------------------------------------------------------------------------------------------------------------------------
def _flying_actor(sac, task, seed=5):
    """a random SAC actor whose throttle bias lifts the drone off, and observation statistics"""
    from fpv_drone_rl_agent_b200 import ppo

    shape = "hover128" if task == 0 else "yaw128"
    m = _actor(sac, shape, seed=seed)
    with torch.no_grad():
        if task == 0:
            m.mu.weight[:3].mul_(0.05)
            m.mu.weight[3].mul_(0.1)
            m.mu.bias.copy_(torch.tensor([0.0, 0.0, 0.0, 0.25]))
    od = SHAPES[shape][0]
    stats = ppo.RunningStats(od, "cuda:0")
    g = torch.Generator().manual_seed(seed)
    stats.mean.copy_(0.1 * torch.randn(od, generator=g))
    stats.inv_std.copy_(0.5 + torch.rand(od, generator=g))
    return sac.PackedSacActor(m, "cuda:0"), stats


def _hand_loop(pkg, sac, packed, stats, cfg, n, seed, clip):
    """sac_actor_forward + QuadXSim.step + episode_record on a sim built as the evaluator builds its own"""
    c = pkg.QxConfig.from_buffer_copy(cfg)
    c.update(auto_reset=0)
    sim = pkg.QuadXSim(n, c, seed=seed, env_id0=0)
    d = sim.device
    obs, act = torch.zeros(n, sim.obs_dim, device=d), torch.zeros(n, sim.act_dim, device=d)
    rew, te, tr = torch.zeros(n, device=d), torch.zeros(n, dtype=torch.uint8, device=d), torch.zeros(n, dtype=torch.uint8, device=d)
    ret, length, end = torch.zeros(n, device=d), torch.zeros(n, dtype=torch.int32, device=d), torch.zeros(n, dtype=torch.int32, device=d)
    n_closed = torch.zeros(1, dtype=torch.int32, device=d)
    norm = (stats.mean.clone(), stats.inv_std.clone())
    sim.reset(obs)
    for step in range(int(c.max_steps) + 2):
        sac.sac_actor_forward(packed, obs, norm=norm, obs_clip=clip, actions=act)
        sim.step(act, obs, rew, te, tr)
        sim.episode_record(ret, length, end, n_closed)
        if step % 16 == 15 and int(n_closed.item()) == n:
            break
    assert int(n_closed.item()) == n
    sim.close()
    return {"return": ret, "length": length, "end": end}


@pytest.mark.parametrize("task,graph", [(0, True), (0, False), (1, True)])
def test_evaluator_records_match_hand_loop(env, task, graph):
    """evaluate_policy with a PackedSacActor: return, length and end flags of every episode bit-identical to the hand loop"""
    import fpv_drone_rl_agent_b200 as pkg

    _lib, ppo, sac = env
    packed, stats = _flying_actor(sac, task)
    cfg = pkg.default_config(task)
    if task == 0:  # spawns spread around (0, 0, 1) and the floor rule off: dome exits at many different steps
        cfg.update(render=1, start_pos=[0, 0, 1.0], spawn_throttle=0.495, spawn_pos_noise=0.8, spawn_yaw_noise=0.4)
    n, seed = 4096, 13
    summary, rec = ppo.evaluate_policy(packed, stats, cfg, n, seed, task=task, obs_clip=10.0, use_cuda_graph=graph)
    ref = _hand_loop(pkg, sac, packed, stats, cfg, n, seed, 10.0)
    for k in ("return", "length", "end"):
        assert torch.equal(rec[k], ref[k]), k
    ln = rec["length"].cpu().numpy()
    print(f"measured SAC evaluation task {task}: mean_reward {summary['mean_reward']:.3f}, lengths {ln.min()}..{ln.max()}")
    assert len(np.unique(ln)) > 3, "the episodes should end at different steps"


def _ppo_artifacts(tmp_path):
    from fpv_drone_rl_agent_b200 import ppo

    tr = ppo.PPOTrainer(ppo.PPOConfig(n_envs=4096, n_steps=16, seed=2, batch_size=16384, n_epochs=2), device="cuda:0")
    tr.learn_iteration()
    tr.save(str(tmp_path / "hover.pt"))
    tr.save_sb3(str(tmp_path / "hover.zip"))
    return tr


def test_ppo_through_sb3_zip_equals_checkpoint(env, tmp_path):
    """A PPO policy and its statistics read back from the SB3 archive evaluate exactly as the trainer's own (what --checkpoint
    flies), in-process and through eval_hover_b200.py."""
    _lib, ppo, sac = env
    tr = _ppo_artifacts(tmp_path)
    arc = sac.load_sb3_zip(str(tmp_path / "hover.zip"), "cuda:0")
    assert arc.algorithm == "PPO"
    stats = sac.obs_stats_from_vecnormalize(arc.vecnormalize, "cuda:0")
    assert torch.equal(stats.mean, tr.rollout.obs_stats.mean) and torch.equal(stats.inv_std, tr.rollout.obs_stats.inv_std)
    packed = arc.pack("cuda:0")
    for name in ("w1", "w2p", "w2v", "w3", "b1", "b2", "b3", "log_std"):
        assert torch.equal(getattr(packed, name), getattr(tr.packed, name)), name
    cfg = tr.sim.cfg
    _, r_zip = ppo.evaluate_policy(packed, stats, cfg, 1024, 1, obs_clip=float(arc.vecnormalize["clip_obs"]))
    _, r_ckpt = ppo.evaluate_policy(tr.packed, tr.rollout.obs_stats, cfg, 1024, 1, obs_clip=tr.cfg.clip_obs)
    for k in ("return", "length", "end"):
        assert torch.equal(r_zip[k], r_ckpt[k]), k
    tr.sim.close()
    outs = []
    for args in (["--checkpoint", str(tmp_path / "hover.pt")], ["--sb3-zip", str(tmp_path / "hover.zip")]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "eval_hover_b200.py"), *args, "--episodes", "1024", "--seed", "1"],
                           cwd=tmp_path, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-4000:]
        outs.append(json.loads(r.stdout.strip().splitlines()[-1]))
    assert outs[1].pop("algorithm") == "PPO"
    assert outs[0] == outs[1]


def test_eval_script_flies_a_sac_archive(env, tmp_path):
    """eval_hover_b200.py --sb3-zip on an SB3-layout SAC archive with --vecnormalize: the summary of evaluate_policy on the
    same actor and statistics, plus "algorithm": "SAC"."""
    from tests.test_sb3_import import _sac_data, _sac_state_dict, _write_archive

    _lib, ppo, sac = env
    sd = _sac_state_dict(seed=7)
    sd["actor.mu.bias"] = torch.tensor([0.0, 0.0, 0.0, 0.3])
    path = _write_archive(tmp_path / "sac_hover.zip", sd, _sac_data())
    g = np.random.default_rng(7)
    vn = {"obs_rms.mean": g.normal(0, 0.1, 20), "obs_rms.var": g.uniform(0.5, 2.0, 20), "obs_rms.count": np.float64(1e6),
          "clip_obs": np.float64(5.0), "epsilon": np.float64(1e-8), "norm_obs": np.bool_(True)}
    np.savez(tmp_path / "vn.npz", **vn)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "eval_hover_b200.py"), "--sb3-zip", path, "--vecnormalize", str(tmp_path / "vn.npz"),
                        "--episodes", "1024", "--seed", "3"], cwd=tmp_path, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out.pop("algorithm") == "SAC"
    arc = sac.load_sb3_zip(path, "cuda:0")
    stats = sac.obs_stats_from_vecnormalize(sac.load_vecnormalize(str(tmp_path / "vn.npz")), "cuda:0")
    summary, _ = ppo.evaluate_policy(arc.pack("cuda:0"), stats, None, 1024, 3, obs_clip=5.0)
    assert out == summary
