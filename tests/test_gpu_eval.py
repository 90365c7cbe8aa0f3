"""qx_episode_record, ppo.PolicyEvaluator / ppo.evaluate_policy, PPOTrainer.evaluate and the evaluation entry points.

The ledger is checked against a host restatement built from the step outputs and qx_get_flags; the evaluator against the
playback loop of test_hover.py:13-27 (one env, deterministic policy, step until done), at a batch size that runs the generic
step kernel and at one that runs the hot kernel.  Both comparisons are exact: the step kernel variants are bitwise equal
(tests/test_gpu_properties.py) and rows of the policy forward are independent."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F_TERM, F_TRUNC, F_OOB, F_FLOOR = 2, 4, 8, 16


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge

    ge.build()
    import fpv_drone_rl_agent_b200 as pkg

    return pkg


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _records(n, d):
    return (torch.zeros(n, device=d), torch.zeros(n, dtype=torch.int32, device=d), torch.zeros(n, dtype=torch.int32, device=d),
            torch.zeros(1, dtype=torch.int32, device=d))


@pytest.mark.parametrize("render", [0, 1])
def test_ledger_matches_host_restatement(pkg, render):
    """4096 hover envs without auto-reset, motor noise on: full throttle in envs [0, 1024) (leaves the dome), a3 = -1 in
    [1024, 2048) (floor rule on step 32; with render = 1 the floor rule is off and they sit until the time limit), U(-1, 1) in
    the rest.  At each env's first step with terminated | truncated the reference takes the length, the fp32 running sum of
    its rewards in step order and the flags word; the records must equal it bit for bit."""
    n = 4096
    cfg = pkg.default_config()
    cfg.update(auto_reset=0, noise=1, render=render)
    sim = pkg.QuadXSim(n, cfg, seed=11 + render)
    d = sim.device
    obs, rew = torch.zeros(n, 20, device=d), torch.zeros(n, device=d)
    te, tr = torch.zeros(n, dtype=torch.uint8, device=d), torch.zeros(n, dtype=torch.uint8, device=d)
    ret, length, end, n_closed = _records(n, d)
    sim.reset(obs)
    rng = np.random.default_rng(render)
    acc = np.zeros(n, np.float32)
    ref_ret, ref_len, ref_end = np.zeros(n, np.float32), np.zeros(n, np.int32), np.zeros(n, np.uint32)
    closed = np.zeros(n, bool)
    for k in range(405):
        a = np.zeros((n, 4), np.float32)
        a[:1024, 3] = 1.0
        a[1024:2048, 3] = -1.0
        a[2048:] = rng.uniform(-1, 1, (n - 2048, 4))
        sim.step(torch.from_numpy(a).to(d), obs, rew, te, tr)
        sim.episode_record(ret, length, end, n_closed)
        r = rew.cpu().numpy()
        ended = (te | tr).cpu().numpy().astype(bool)
        flags = sim.flags()
        live = ~closed
        acc[live] = acc[live] + r[live]
        new = live & ended
        ref_ret[new], ref_len[new], ref_end[new] = acc[new], k + 1, flags[new]
        closed |= new
    assert closed.all()
    assert int(n_closed.item()) == n
    got_ret, got_len, got_end = ret.cpu().numpy(), length.cpu().numpy(), end.cpu().numpy().view(np.uint32)
    assert np.array_equal(got_len, ref_len)
    assert np.array_equal(got_end, ref_end)
    assert np.array_equal(got_ret.view(np.int32), ref_ret.view(np.int32)), float(np.abs(got_ret - ref_ret).max())
    assert (got_end != 0).all() and ((got_end & (F_TERM | F_TRUNC)) != 0).all()
    assert ((got_end[:1024] & F_OOB) != 0).all()  # full throttle leaves the dome
    if render:
        assert (got_len[1024:2048] == cfg.max_steps + 2).all()
        assert ((got_end[1024:2048] & (F_TERM | F_TRUNC)) == F_TRUNC).all()
    else:
        assert (got_len[1024:2048] == cfg.floor_grace_steps + 2).all()
        assert ((got_end[1024:2048] & (F_TERM | F_FLOOR)) == F_TERM | F_FLOOR).all()
    sim.close()


def _policy(task, seed=3):
    """A random policy with a strong action head (the default 0.01-gain head barely moves the drone), a throttle bias that
    lifts the drone off, and non-trivial observation statistics."""
    from fpv_drone_rl_agent_b200 import ppo

    od, ad = (20, 4) if task == 0 else (12, 1)
    torch.manual_seed(seed)
    model = ppo.ActorCritic(od, ad).cuda()
    with torch.no_grad():
        model.mu.weight.mul_(40.0)
        if ad == 4:  # hover: gentle rate commands and a throttle above hover that depends on the observation
            model.mu.weight[:3].mul_(0.1)
            model.mu.bias.copy_(torch.tensor([0.0, 0.0, 0.0, 0.2]))
    stats = ppo.RunningStats(od, "cuda:0")
    g = torch.Generator().manual_seed(seed)
    stats.mean.copy_(0.1 * torch.randn(od, generator=g))
    stats.inv_std.copy_(0.5 + torch.rand(od, generator=g))
    return ppo.PackedPolicy(model, "cuda:0"), stats


def _playback(pkg, packed, stats, cfg, seed, env_id):
    """test_hover.py's loop for env `env_id` of a batch: its own one-env sim, predict(deterministic=True) on one row, step
    until done; the return summed in fp32 in step order."""
    from fpv_drone_rl_agent_b200 import ppo

    sim = pkg.QuadXSim(1, cfg, seed=seed, env_id0=env_id)
    d = sim.device
    obs, act = torch.zeros(1, sim.obs_dim, device=d), torch.zeros(1, sim.act_dim, device=d)
    rew, te, tr = torch.zeros(1, device=d), torch.zeros(1, dtype=torch.uint8, device=d), torch.zeros(1, dtype=torch.uint8, device=d)
    sim.reset(obs)
    total, steps = np.float32(0.0), 0
    while True:
        ppo.policy_forward(packed, obs, norm=(stats.mean, stats.inv_std), obs_clip=10.0, deterministic=True, env_actions=act)
        sim.step(act, obs, rew, te, tr)
        steps += 1
        total = np.float32(total + np.float32(rew.item()))
        if te.item() or tr.item():
            break
        assert steps <= cfg.max_steps + 2
    flags = int(sim.flags()[0])
    sim.close()
    return total, steps, flags


@pytest.mark.parametrize("task", [0, 1])
def test_evaluator_matches_single_env_playback(pkg, task):
    from fpv_drone_rl_agent_b200 import ppo

    packed, stats = _policy(task)
    cfg = pkg.default_config(task)
    if task == 0:  # spawns spread around (0, 0, 1) and the floor rule off: dome exits at many different steps
        cfg.update(render=1, start_pos=[0, 0, 1.0], spawn_throttle=0.495, spawn_pos_noise=0.8, spawn_yaw_noise=0.4)
    seed = 21
    ids = [0, 1, 2, 37, 100, 255, 300, 511]
    play_cfg = pkg.QxConfig.from_buffer_copy(cfg)
    play_cfg.update(auto_reset=0)
    ref = [_playback(pkg, packed, stats, play_cfg, seed, i) for i in ids]
    for n in (512, 65536):  # 65 536 hover envs run the hot step kernel
        summary, rec = ppo.evaluate_policy(packed, stats, cfg, n, seed, task=task)
        r, ln, e = rec["return"].cpu().numpy(), rec["length"].cpu().numpy(), rec["end"].cpu().numpy()
        for i, (tot, steps, flags) in zip(ids, ref):
            assert (ln[i], e[i]) == (steps, flags), (n, i, ln[i], steps, e[i], flags)
            assert r[i].view(np.int32) == tot.view(np.int32), (n, i, float(r[i]), float(tot))
        assert summary["n_episodes"] == n and summary["mean_ep_length"] == pytest.approx(float(ln.mean()))
        assert summary["mean_reward"] == pytest.approx(float(r.astype(np.float64).mean()))
        assert summary["std_reward"] == pytest.approx(float(r.astype(np.float64).std()))
        assert summary["success_rate"] == pytest.approx(float((((e & F_TRUNC) != 0) & ((e & F_TERM) == 0)).mean()))
        assert summary["floor_rate"] == pytest.approx(float(((e & F_FLOOR) != 0).mean()))
        assert summary["oob_rate"] == pytest.approx(float(((e & F_OOB) != 0).mean()))
        if n == 512 and task == 0:
            assert len(np.unique(ln)) > 5, "the episodes should end at many different steps"


def _same(a, b):
    return all(torch.equal(a[k], b[k]) for k in ("return", "length", "end"))


def test_graph_chunks_repeats_and_seeds(pkg):
    from fpv_drone_rl_agent_b200 import ppo

    packed, stats = _policy(0, seed=5)
    cfg = pkg.default_config()
    base = ppo.PolicyEvaluator(packed, stats, cfg, 4096, seed=9)
    s1, r1 = base.evaluate()
    s2, r2 = base.evaluate()
    assert _same(r1, r2) and s1 == s2
    _, r_eager = ppo.evaluate_policy(packed, stats, cfg, 4096, 9, use_cuda_graph=False)
    assert _same(r1, r_eager)
    _, r_chunk = ppo.evaluate_policy(packed, stats, cfg, 4096, 9, chunk=7)
    assert _same(r1, r_chunk)
    _, r_seed = ppo.evaluate_policy(packed, stats, cfg, 4096, 10)
    assert not torch.equal(r1["return"], r_seed["return"])
    # the statistics are read at evaluate(), not when the evaluator was built
    stats.mean.add_(0.05)
    _, r3 = base.evaluate()
    assert not torch.equal(r1["return"], r3["return"])
    base.close()


def _training_state(tr):
    """Everything the next training iteration reads: every tensor of the rollout engine, its statistics, the fused updater and
    the packed policy, the model, the env state and Monitor sums, the minibatch generator and torch's random streams."""
    def bits(t):  # compared as bytes: a NaN that stays a NaN is unchanged
        return t.detach().reshape(-1).contiguous().view(torch.uint8).cpu()

    out = {}
    for name, obj in (("rollout", tr.rollout), ("obs_stats", tr.rollout.obs_stats), ("ret_stats", tr.rollout.ret_stats),
                      ("fused", tr.fused), ("packed", tr.packed)):
        for k, v in vars(obj).items():
            if torch.is_tensor(v):
                out[f"{name}.{k}"] = bits(v)
    out.update({f"model.{k}": bits(v) for k, v in tr.model.state_dict().items()})
    out.update({f"sim.{k}": bits(torch.from_numpy(v.copy().view(np.int32))) for k, v in tr.sim.get_state().items()})
    out["sim.episode_stats"] = bits(torch.tensor(tr.sim.episode_stats(clear=False), dtype=torch.float64))
    out["gen"], out["cpu_rng"], out["cuda_rng"] = tr.gen.get_state(), torch.get_rng_state(), torch.cuda.get_rng_state()
    out["counters"] = torch.tensor([tr.num_timesteps, tr._iteration, tr.fused.adam_steps])
    return out


def test_trainer_evaluate_leaves_training_unchanged(pkg):
    """PPOTrainer.evaluate between iterations reads the policy and the statistics and writes nothing of the training loop.
    Two training runs are not bitwise reproducible by themselves -- the fused update and the Monitor sums reduce with float
    atomics across blocks (tests/test_gpu_update.py::test_checkpoint_resume allows 5e-5) -- so the test compares the whole
    state the next iteration reads, bit for bit, before and after each evaluation: with it equal, an iteration after an
    evaluation computes what it would have computed without it."""
    from fpv_drone_rl_agent_b200 import ppo

    tr = ppo.PPOTrainer(ppo.PPOConfig(n_envs=4096, n_steps=16, seed=2, batch_size=16384, n_epochs=2), device="cuda:0")
    evals = []
    for _ in range(3):
        tr.learn_iteration()
        torch.cuda.synchronize()
        before = _training_state(tr)
        evals.append(tr.evaluate(1024))
        torch.cuda.synchronize()
        after = _training_state(tr)
        assert before.keys() == after.keys() and len(before) > 40
        changed = [k for k in before if not torch.equal(before[k], after[k])]
        assert not changed, changed
    assert [e[0]["n_episodes"] for e in evals] == [1024] * 3
    assert evals[0][0] != evals[2][0]  # the evaluator follows the weights as they train
    assert tr.evaluate(1024)[0] == evals[2][0]  # and repeats itself on unchanged weights
    tr.sim.close()


def test_record_arguments(pkg):
    from fpv_drone_rl_agent_b200 import ppo

    L = pkg._lib.lib()
    cfg = pkg.default_config()
    cfg.update(auto_reset=0)
    sim = pkg.QuadXSim(256, cfg, seed=1)
    auto = pkg.QuadXSim(256, pkg.default_config(), seed=1)
    ret, length, end, n_closed = _records(256, sim.device)
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    bufs = [_p(ret), _p(length), _p(end), _p(n_closed)]
    n0 = L.qx_launch_count()
    assert L.qx_episode_record(None, *bufs, s) == -1
    assert L.qx_episode_record(auto._h, *bufs, s) == -1
    assert b"auto_reset" in L.qx_last_error()
    for k in range(4):
        args = list(bufs)
        args[k] = None
        assert L.qx_episode_record(sim._h, *args, s) == -1
    assert L.qx_launch_count() == n0
    assert L.qx_episode_record(sim._h, *bufs, s) == 0 and L.qx_launch_count() == n0 + 1
    with pytest.raises(ValueError):
        sim.episode_record(ret, length.float(), end, n_closed)
    # yaw handles keep a ledger too
    ycfg = pkg.default_config(pkg.QX_TASK_YAW)
    ycfg.update(auto_reset=0)
    ysim = pkg.QuadXSim(256, ycfg, seed=1)
    assert L.qx_episode_record(ysim._h, *bufs, s) == 0
    torch.cuda.synchronize()
    # a policy for the other task, statistics of the wrong width, a config of the other task
    hover_pol, hover_stats = _policy(0)
    yaw_pol, _ = _policy(1)
    with pytest.raises(ValueError, match="obs_dim"):
        ppo.PolicyEvaluator(hover_pol, None, pkg.default_config(pkg.QX_TASK_YAW), 64, task=pkg.QX_TASK_YAW)
    with pytest.raises(ValueError, match="obs_dim"):
        ppo.PolicyEvaluator(yaw_pol, None, None, 64, task=pkg.QX_TASK_HOVER)
    with pytest.raises(ValueError, match="obs_stats"):
        ppo.PolicyEvaluator(yaw_pol, hover_stats, None, 64, task=pkg.QX_TASK_YAW)
    with pytest.raises(ValueError, match="task"):
        ppo.PolicyEvaluator(hover_pol, None, pkg.default_config(pkg.QX_TASK_YAW), 64, task=pkg.QX_TASK_HOVER)
    for h in (sim, auto, ysim):
        h.close()


def test_entry_points(pkg, tmp_path):
    """train_hover_b200.py --eval-every 1 logs an evaluation per iteration; eval_hover_b200.py on the hover.pt it saved prints
    the summary of the trainer's last evaluation (same weights, episodes and seed)."""
    env = dict(os.environ)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "train_hover_b200.py"), "--envs", "4096", "--steps", "16", "--iters", "2",
                        "--batch", "16384", "--eval-every", "1", "--eval-episodes", "1024", "--json", "log.json",
                        "--save-path", str(tmp_path / "ckpt")], cwd=tmp_path, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    log = json.load(open(tmp_path / "log.json"))
    assert len(log) == 2 and all("eval" in e for e in log)
    keys = {"mean_reward", "std_reward", "mean_ep_length", "success_rate", "floor_rate", "oob_rate", "n_episodes", "steps"}
    assert all(set(e["eval"]) == keys and e["eval"]["n_episodes"] == 1024 for e in log)
    assert r.stdout.count("eval ") == 2
    r2 = subprocess.run([sys.executable, os.path.join(ROOT, "eval_hover_b200.py"), "--checkpoint", str(tmp_path / "hover.pt"),
                         "--episodes", "1024", "--seed", "1"], cwd=tmp_path, env=env, capture_output=True, text=True, timeout=900)
    assert r2.returncode == 0, r2.stderr[-4000:]
    assert json.loads(r2.stdout.strip().splitlines()[-1]) == log[-1]["eval"]
