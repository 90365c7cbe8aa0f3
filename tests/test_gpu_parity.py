"""GPU: the CUDA env-step path, called through the C-ABI, against the oracle and
the committed golden vectors.

Tolerances (north star: fp32 trajectories within 1e-3 relative over 500 control
steps; flags exact):
  * rigid-body / motor state after 500 steps of the SAME action sequence:
    |cuda - oracle| <= 1e-3 * max(full scale, |oracle|), full scale = 3 m (the
    flight dome, hover.py:37) for position and 1 for quaternion, m/s, rad/s and
    throttle.  The actions are computed from the oracle's state, so the CUDA
    trajectory is open loop and fp32 rounding of the attitude integrates twice
    into position; the measured worst case is printed by the test.
  * observation columns not produced by the camera: 2e-3 absolute (the finite
    difference of Euler angles is divided by 0.025, hover.py:230)
  * camera columns vs the *rasterised* golden frames: the analytic-vs-pixel
    bounds measured in tests/test_oracle_golden.py (1.5 px centre, 10 % area,
    one pixel row/column in the bbox ratio); vs the analytic oracle: 2e-3
  * reward: vs analytic oracle 5e-3; vs rasterised golden 0.45 (sum of the
    camera bounds, hover.py:305-317)
"""
import os

import numpy as np
import pytest
import torch

from tests.util import NONVISION_COLS, VISION_COLS, ForkAccount, kernel_state_arrays, oracle_to_kernel_state

pytestmark = pytest.mark.gpu

HOVER_THR = float(np.sqrt(0.1 * 9.81 / 4.0))  # pwm at which thrust = weight (cf2x.yaml:2, cf2x.urdf:10)


def _close(a, b, tol, what, scale=1.0):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if a.size == 0:
        return 0.0
    err = np.abs(a - b) / np.maximum(scale, np.abs(b))
    assert err.max() <= tol, f"{what}: max rel err {err.max():.3e} at {np.unravel_index(err.argmax(), err.shape)}"
    return err.max()


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge

    ge.build()
    import fpv_drone_rl_agent_b200 as pkg

    return pkg


_VARIANTS = {
    "generic": {"QX_HOT": "0"},                                                    # quadx_step_kernel: what small batches, step_k, yaw and the flight modes run
    "hot_paired_merged": {"QX_HOT": "1", "QX_LANES": "4", "QX_MERGED": "1"},        # the large-batch default: one env per thread, components paired on FFMA2 / FMUL2 / FADD2, one launch for step + reset
    "hot_scalar_two_launches": {"QX_HOT": "1", "QX_LANES": "1", "QX_MERGED": "0"},  # lean scalar step kernel + separate reset-queue launch
    "hot_two_envs_packed": {"QX_HOT": "1", "QX_LANES": "2", "QX_MERGED": "1"},      # two envs per thread on FFMA2 / FMUL2 / FADD2
}


@pytest.fixture(autouse=True, params=list(_VARIANTS))
def kernel_variant(request, monkeypatch):
    """Every parity test runs through each env-step kernel variant (the variables are read at qx_create)."""
    for k, v in _VARIANTS[request.param].items():
        monkeypatch.setenv(k, v)
    return request.param


def _airborne(pkg, n, seed, noise, auto_reset=0, max_steps=400):
    """CUDA sim + oracle in the airborne configuration of SURVEY 8d C2."""
    from oracle.hover_oracle import HoverConfig, HoverVecOracle
    from oracle.quadx_model import QuadXParams

    cfg = pkg.default_config()
    cfg.update(start_pos=[0, 0, 1.0], spawn_throttle=HOVER_THR, reset_idle_steps=0, auto_reset=auto_reset, noise=int(noise), max_steps=max_steps)
    sim = pkg.QuadXSim(n, cfg, seed=seed)
    orc = HoverVecOracle(
        n, QuadXParams(), HoverConfig(start_pos=(0, 0, 1.0), spawn_throttle=HOVER_THR, reset_idle_steps=0, max_steps=max_steps),
        seed=seed, auto_reset=bool(auto_reset), noise=noise,
    )
    return sim, orc


class _Bufs:
    def __init__(self, sim):
        n, d = sim.n, sim.device
        self.obs = torch.zeros(n, 20, device=d)
        self.rew = torch.zeros(n, device=d)
        self.te = torch.zeros(n, dtype=torch.uint8, device=d)
        self.tr = torch.zeros(n, dtype=torch.uint8, device=d)
        self.tobs = torch.zeros(n, 20, device=d)

    def step(self, sim, a):
        sim.step(torch.as_tensor(a, dtype=torch.float32, device=sim.device).contiguous(), self.obs, self.rew, self.te, self.tr, self.tobs)
        torch.cuda.synchronize()
        return self.obs.cpu().numpy(), self.rew.cpu().numpy(), self.te.cpu().numpy().astype(bool), self.tr.cpu().numpy().astype(bool)


@pytest.mark.parametrize("noise", [False, True])
def test_free_flight_trajectory_500_steps(pkg, noise):
    """500 control steps of free flight under a feedback test policy: state
    trajectories within 1e-3 relative of the float64 oracle, flags identical."""
    from oracle.test_policy import hover_actions

    n = 256
    sim, orc = _airborne(pkg, n, seed=42, noise=noise, max_steps=1000)  # no time limit inside the 500 steps
    b = _Bufs(sim)
    sim.reset(b.obs)
    obs_o = orc.reset()
    _close(b.obs.cpu().numpy(), obs_o, 2e-3, "reset obs")
    rng = np.random.default_rng(0)
    tgt = np.stack([rng.uniform(-1, 1, n), rng.uniform(-1, 1, n), rng.uniform(0.6, 1.6, n)], 1)
    worst, flips, seen = {}, 0, 0
    for k in range(500):
        a = hover_actions(orc.st.aviary_state(), tgt, rng, 0.1).astype(np.float32)
        o, r, te, tr = b.step(sim, a)
        o2, r2, te2, tr2, _ = orc.step(a.astype(np.float64))
        live = ~(te2 | tr2)
        assert np.array_equal(te, te2) and np.array_equal(tr, tr2), f"flags differ at step {k}"
        if k % 25 == 24 or k == 499:
            pos, quat, vel, om, thr = kernel_state_arrays(sim.get_state())
            sgn = np.sign((quat * orc.st.quat).sum(1, keepdims=True))
            for name, x, y, sc in (("pos", pos, orc.st.pos, 3.0), ("quat", quat * sgn, orc.st.quat, 1.0), ("vel", vel, orc.st.vel, 1.0),
                                   ("omega", om, orc.st.omega, 1.0), ("thr", thr, orc.st.thr, 1.0)):
                worst[name] = max(worst.get(name, 0.0), _close(x[live], y[live], 1e-3, f"{name} @ step {k}", sc))
        _close(o[live][:, NONVISION_COLS], o2[live][:, NONVISION_COLS], 2e-3, f"obs @ step {k}")
        # the bbox ratio is a quotient of pixel counts (hover.py:209-213): a corner within fp32 rounding of a pixel
        # boundary flips one count, so the reward is compared where the camera columns agree
        same = live & (o[:, 13] == o2[:, 13]) & (np.abs(o[:, 14] - o2[:, 14]) < 1e-4)
        flips += int((live & ~same).sum())
        seen += int(live.sum())
        _close(r[same], r2[same], 5e-3, f"reward @ step {k}")
    assert flips <= 0.01 * seen, (flips, seen)
    assert (~(orc.terminated | orc.truncated)).sum() > 0.9 * n  # the envs really flew all 500 steps
    print(f"noise={noise}: worst state error / full scale over 500 steps:", {k: f"{v:.2e}" for k, v in worst.items()})


def test_vision_columns_match_analytic_oracle(pkg):
    from oracle.test_policy import hover_actions

    n = 512
    sim, orc = _airborne(pkg, n, seed=3, noise=True)
    b = _Bufs(sim)
    sim.reset(b.obs)
    orc.reset()
    rng = np.random.default_rng(5)
    tgt = np.stack([rng.uniform(-2, 2, n), rng.uniform(-2, 2, n), rng.uniform(0.4, 2.2, n)], 1)
    n_vis = mism = tot = 0
    for k in range(120):
        a = hover_actions(orc.st.aviary_state(), tgt, rng, 0.1).astype(np.float32)
        o, r, te, tr = b.step(sim, a)
        o2, r2, te2, tr2, _ = orc.step(a.astype(np.float64))
        live = ~(te2 | tr2)
        same = (o[:, 13] == o2[:, 13]) & live
        mism += int((~same & live).sum())
        tot += int(live.sum())
        n_vis += int((o2[:, 13] > 0.5).sum())
        # ratio is a quotient of pixel counts: a corner within fp32 rounding of a pixel boundary may flip one count
        cols = [7, 8, 9, 10, 11, 12]
        _close(o[same][:, cols], o2[same][:, cols], 2e-3, f"vision @ {k}")
        flip = np.abs(o[same][:, 14] - o2[same][:, 14]) > 1e-4
        assert flip.mean() < 0.01
    assert mism / tot < 1e-3 and n_vis > 0.3 * tot


GOLDEN = ["fly_quiet", "fly_noisy", "floor", "dome", "render_idle", "agent_hz60"]


@pytest.mark.parametrize("name", GOLDEN)
def test_golden_reference_trajectories(pkg, golden_dir, name):
    """Replay the action sequences recorded with the reference's own hover.py in
    the loop through the gymnasium-shaped facade; compare every output."""
    g = np.load(os.path.join(golden_dir, f"hover_ref_{name}.npz"))
    render = bool(g["render"]) if "render" in g.files else False  # hover.py:283: rendering switches the floor rule off
    agent_hz = int(g["agent_hz"]) if "agent_hz" in g.files else 40  # hover.py:14,24-25
    env = pkg.QuadXHoverEnv(agent_hz=agent_hz, render=render, seed=int(g["seed"]), noise=int(bool(g["noise"])))
    # the facade creates env id 0; golden env ids other than 0 need the raw sim
    if int(g["env_id"]) != 0:
        env.sim.close()
        cfg = pkg.default_config()
        cfg.update(auto_reset=0, noise=int(bool(g["noise"])))
        env.sim = pkg.QuadXSim(1, cfg, seed=int(g["seed"]), env_id0=int(g["env_id"]))
    ep = -1
    vis_mismatch = 0
    for k in range(g["actions"].shape[0]):
        if g["episode_start"][k]:
            ep += 1
            obs, info = env.reset()
            _close(obs[NONVISION_COLS], g["reset_obs"][ep][NONVISION_COLS], 2e-3, "reset obs")
            assert info == {"out_of_bounds": False, "collision": False, "env_complete": False, "on_floor": False}
        o, r, te, tr, info = env.step(g["actions"][k])
        assert te == bool(g["terminated"][k]) and tr == bool(g["truncated"][k]), f"flags at step {k}"
        _close(o[NONVISION_COLS], g["obs"][k][NONVISION_COLS], 2e-3, f"obs step {k}")
        go = g["obs"][k]
        if o[13] == go[13]:
            if go[13] > 0.5:
                assert np.abs(o[7:9] - go[7:9]).max() * 64 <= 1.5
                assert abs(o[11] - go[11]) <= 0.10 * go[11]
                assert abs(o[14] - go[14]) <= 0.35
            assert abs(r - g["reward"][k]) <= 0.45, f"reward step {k}: {r} vs {g['reward'][k]}"
        else:
            vis_mismatch += 1
        st = env.sim.get_state()
        s_pos_ok = np.abs(np.array([st["px"][0], st["py"][0], st["pz"][0]]) - g["state"][k][3]).max()
        assert s_pos_ok < 0.1  # true pose vs one-sub-step-stale snapshot: h * |v|, up to 12 m/s in the dome scenario
    assert vis_mismatch <= 2
    if name == "floor":
        assert info["on_floor"] and not info["out_of_bounds"]
    if name == "dome":
        assert info["out_of_bounds"]
    if name == "render_idle":
        assert not info["on_floor"] and not bool(g["terminated"].any())  # 40 steps on the floor, never terminated
    env.close()


def test_auto_reset_semantics(pkg):
    """SB3 VecEnv contract: reward/flags of the terminal step, obs of the next
    episode, terminal observation on the side, Monitor statistics."""
    from oracle.hover_oracle import HoverVecOracle

    n = 96
    env = pkg.QuadXHoverVecEnv(n, seed=5)
    orc = HoverVecOracle(n, seed=5, noise=True)
    _close(env.reset().cpu().numpy(), orc.reset(), 2e-3, "reset")
    a = np.tile(np.array([[0.0, 0.0, 0.0, -1.0]], np.float32), (n, 1))
    for k in range(70):
        o, r, d, infos = env.step(torch.as_tensor(a))
        o2, r2, te2, tr2, info2 = orc.step(a.astype(np.float64))
        assert np.array_equal(d.cpu().numpy(), te2 | tr2)
        _close(r.cpu().numpy(), r2, 5e-3, f"reward {k}")
        _close(o.cpu().numpy(), o2, 2e-3, f"obs {k}")
        if d.any():
            assert k in (31, 63)
            for i in range(n):
                assert infos[i]["TimeLimit.truncated"] is False and infos[i]["episode"]["l"] == 32
                _close(infos[i]["terminal_observation"], info2["terminal_obs"][i], 2e-3, "terminal obs")
    s, l, c = env.episode_stats()
    assert c == 2 * n and l == 64 * n and abs(s - orc.sum_ret) < 1e-3 * abs(orc.sum_ret)
    env.close()


def test_truncation_through_vec_env(pkg):
    """A hovering env runs into the 402-step time limit: TimeLimit.truncated is set."""
    env = pkg.QuadXHoverVecEnv(8, seed=1, start_pos=[0, 0, 1.0], spawn_throttle=HOVER_THR, reset_idle_steps=0, noise=0)
    env.reset()
    a = torch.zeros(8, 4, device=env.device)
    a[:, 3] = 2 * HOVER_THR - 1
    lengths = []
    for k in range(410):
        o, r, d, infos = env.step(a)
        if d.any():
            lengths.append(k + 1)
            assert all(i["TimeLimit.truncated"] and i["episode"]["l"] == 402 for i in infos)
    assert lengths == [402]
    env.close()


def test_host_and_device_entry_points_agree(pkg):
    sim_d, _ = _airborne(pkg, 64, seed=9, noise=True, auto_reset=1)
    sim_h, _ = _airborne(pkg, 64, seed=9, noise=True, auto_reset=1)
    b = _Bufs(sim_d)
    sim_d.reset(b.obs)
    torch.cuda.synchronize()
    assert np.array_equal(b.obs.cpu().numpy(), sim_h.reset_host())
    rng = np.random.default_rng(1)
    for k in range(20):
        a = rng.uniform(-1, 1, (64, 4)).astype(np.float32)
        o, r, te, tr = b.step(sim_d, a)
        o2, r2, te2, tr2, _ = sim_h.step_host(a)
        assert np.array_equal(o, o2) and np.array_equal(r, r2) and np.array_equal(te, te2) and np.array_equal(tr, tr2)


def test_state_roundtrip_and_oracle_injection(pkg):
    """qx_set_state(oracle state) then one step == oracle step (local error only)."""
    from oracle.test_policy import hover_actions

    n = 128
    sim, orc = _airborne(pkg, n, seed=11, noise=True)
    b = _Bufs(sim)
    sim.reset(b.obs)
    orc.reset()
    rng = np.random.default_rng(2)
    tgt = np.stack([rng.uniform(-1, 1, n), rng.uniform(-1, 1, n), rng.uniform(0.6, 1.6, n)], 1)
    flips = 0
    for k in range(60):
        a = hover_actions(orc.st.aviary_state(), tgt, rng, 0.2).astype(np.float32)
        sim.set_state(oracle_to_kernel_state(orc))
        s = sim.get_state()
        assert np.array_equal(s["step_count"], orc.step_count.astype(np.int32))
        o, r, te, tr = b.step(sim, a)
        o2, r2, te2, tr2, _ = orc.step(a.astype(np.float64))
        pos, quat, vel, om, thr = kernel_state_arrays(sim.get_state())
        _close(pos, orc.st.pos, 2e-6, "pos")
        _close(vel, orc.st.vel, 2e-5, "vel")
        _close(om, orc.st.omega, 2e-4, "omega")
        _close(thr, orc.st.thr, 1e-5, "thr")
        # hover.py:209-213: the bbox ratio is a quotient of pixel counts, so a corner within fp32 rounding of a pixel boundary
        # moves ratio and reward by one pixel's worth; such steps are counted (and bounded below), the rest must agree
        same = (o[:, 13] == o2[:, 13]) & (np.abs(o[:, 14] - o2[:, 14]) < 1e-4)
        flips += int((~same).sum())
        _close(r[same], r2[same], 2e-3, "reward")
    assert flips <= 0.005 * 60 * n, flips


@pytest.mark.parametrize("n", [1, 31, 129, 1000])
def test_ragged_batch_sizes_and_masked_reset(pkg, n):
    """Edge cases: batch sizes that are not a multiple of the 128-thread block (incl. a single env), masked resets
    (qx_reset with a mask touches only the selected envs), and get/set-state round trips."""
    from oracle.hover_oracle import HoverVecOracle

    env = pkg.QuadXHoverVecEnv(n, seed=21)
    orc = HoverVecOracle(n, seed=21, noise=True)
    _close(env.reset().cpu().numpy(), orc.reset(), 2e-3, "reset")
    rng = np.random.default_rng(n)
    for k in range(12):
        a = rng.uniform(-1, 1, (n, 4)).astype(np.float32)
        a[:, :3] *= 0.2  # moderate rates and a clean lift-off: floor contact (a sticky plane) is discontinuous, and a
        a[:, 3] = 0.25 + 0.05 * a[:, 3]  # drone scraping along it amplifies fp32-vs-fp64 rounding
        o, r, d, _ = env.step(torch.as_tensor(a))
        o2, r2, te2, tr2, _ = orc.step(a.astype(np.float64))
        _close(o.cpu().numpy()[:, NONVISION_COLS], o2[:, NONVISION_COLS], 2e-3, f"obs {k}")
        assert np.array_equal(d.cpu().numpy(), te2 | tr2)
    # masked reset: only the selected envs change
    before = env.sim.get_state()
    mask = np.zeros(n, bool)
    mask[:: max(1, n // 3)] = True
    obs = torch.full((n, 20), -7.0, device=env.device)
    env.sim.reset(obs, torch.as_tensor(mask, device=env.device))
    torch.cuda.synchronize()
    after = env.sim.get_state()
    o_ref = orc.reset(mask)
    assert np.all(obs.cpu().numpy()[~mask] == -7.0)
    _close(obs.cpu().numpy()[mask][:, NONVISION_COLS], o_ref[mask][:, NONVISION_COLS], 2e-3, "masked reset obs")
    for key in ("px", "pz", "thr0", "step_count", "prev_a3"):
        assert np.array_equal(before[key][~mask], after[key][~mask]), key
    assert np.all(after["step_count"][mask] == 0)
    assert np.array_equal(after["prev_a3"][mask], before["prev_a3"][mask])  # hover.py:31,357: prev_action survives reset
    # state round trip is the identity
    env.sim.set_state(after)
    again = env.sim.get_state()
    for key in after:
        assert np.array_equal(after[key], again[key], equal_nan=True), key
    env.close()


def test_bf16_obs_into_strided_policy_buffer(pkg):
    """The env writes bf16 observations straight into a wider policy input buffer (row stride 32)."""
    n = 300
    sim_a, _ = _airborne(pkg, n, seed=2, noise=True, auto_reset=1)
    sim_b, _ = _airborne(pkg, n, seed=2, noise=True, auto_reset=1)
    buf = torch.zeros(n, 32, dtype=torch.bfloat16, device=sim_a.device)
    ref = torch.zeros(n, 20, device=sim_a.device)
    rew = torch.zeros(n, device=sim_a.device); te = torch.zeros(n, dtype=torch.uint8, device=sim_a.device); tr = torch.zeros_like(te)
    sim_a.reset(buf); sim_b.reset(ref)
    a = torch.rand(n, 4, device=sim_a.device) * 0.4 - 0.2
    for k in range(5):
        sim_a.step(a, buf, rew, te, tr); sim_b.step(a, ref, rew, te, tr)
    torch.cuda.synchronize()
    assert torch.equal(buf[:, :20].float(), ref.to(torch.bfloat16).float()) and torch.all(buf[:, 20:] == 0)


def test_nonfinite_state_is_contained(pkg):
    """Failure containment: an env whose state turns NaN / inf is terminated (like an out-of-bounds flight), counted and
    re-created by the auto-reset; its neighbours in the batch are untouched."""
    n = 256
    a = torch.zeros(n, 4, device="cuda")
    a[:, 3] = 2 * HOVER_THR - 1
    envs = [pkg.QuadXHoverVecEnv(n, seed=8, infos=False, noise=0) for _ in range(2)]
    for e in envs:
        e.reset()
        e.step(a)
    st = envs[0].sim.get_state()
    bad = np.zeros(n, bool)
    bad[[3, 64, 200]] = True
    st["vx"][3] = np.nan
    st["qw"][64] = np.inf
    st["wbz"][200] = np.nan  # (an infinite rate would simply be caught by the +-100 velocity clamp)
    envs[0].sim.set_state(st)
    o0, r0, d0, _ = envs[0].step(a)
    o1, r1, d1, _ = envs[1].step(a)
    torch.cuda.synchronize()
    assert envs[0].sim.nonfinite_count() == 3 and envs[1].sim.nonfinite_count() == 0
    assert np.array_equal(d0.cpu().numpy(), bad) and not d1.any()
    assert torch.isfinite(o0).all() and torch.isfinite(r0).all()
    assert torch.equal(o0[~torch.as_tensor(bad)], o1[~torch.as_tensor(bad)]) and torch.equal(r0[~torch.as_tensor(bad)], r1[~torch.as_tensor(bad)])
    assert (r0[torch.as_tensor(bad)] < -90).all()
    for k in range(3):
        o0, r0, d0, _ = envs[0].step(a)
    assert torch.isfinite(o0).all() and envs[0].sim.nonfinite_count() == 3
    for e in envs:
        e.close()


def test_gym_api_conformance(pkg):
    """What SB3's check_env (yaw.py:217) asserts about a gymnasium env, for both single-env facades: spaces, dtypes,
    reset -> (obs, info), step -> (obs, float, bool, bool, dict), observations inside the observation space."""
    for make, od, ad in ((lambda: pkg.QuadXHoverEnv(seed=1), 20, 4), (lambda: pkg.DroneEnv(seed=1), 12, 1)):
        env = make()
        assert env.action_space.shape == (ad,) and env.observation_space.shape == (od,)
        assert np.all(env.action_space.low == -1) and np.all(env.action_space.high == 1)
        obs, info = env.reset(seed=0)
        assert isinstance(info, dict) and obs.shape == (od,) and np.all(np.isfinite(obs))
        rng = np.random.default_rng(0)
        for _ in range(5):
            a = env.action_space.sample(rng)
            assert env.action_space.contains(a)
            out = env.step(a)
            assert len(out) == 5
            obs, r, te, tr, info = out
            assert obs.shape == (od,) and isinstance(r, float) and isinstance(te, bool) and isinstance(tr, bool) and isinstance(info, dict)
            assert np.all(obs >= env.observation_space.low - 1e-6) and np.all(obs <= env.observation_space.high + 1e-6)
        if od == 20:
            assert obs.dtype == np.float64 and set(info) == {"out_of_bounds", "collision", "env_complete", "on_floor"}  # hover.py:53-57,70
        env.close()
    # the env refuses wrong-shaped device buffers loudly instead of corrupting memory
    sim = pkg.QuadXSim(64)
    with pytest.raises(ValueError):
        sim.step(torch.zeros(63, 4, device="cuda"), None, torch.zeros(64, device="cuda"), torch.zeros(64, dtype=torch.uint8, device="cuda"),
                 torch.zeros(64, dtype=torch.uint8, device="cuda"))
    # an observation view with fewer than obs_dim columns: its row stride leaves room for 20, but the view ends before that
    wide = torch.full((64, 24), 7.0, device="cuda")
    for narrow in (wide[:, :19], wide[:, :4]):
        with pytest.raises(ValueError, match="obs"):
            sim.reset(narrow)
        with pytest.raises(ValueError, match="obs"):
            sim.step(torch.zeros(64, 4, device="cuda"), narrow, torch.zeros(64, device="cuda"), torch.zeros(64, dtype=torch.uint8, device="cuda"),
                     torch.zeros(64, dtype=torch.uint8, device="cuda"))
    torch.cuda.synchronize()
    assert torch.all(wide == 7.0)
    sim.reset(wide[:, :20])  # the full width at row stride 24 is accepted and leaves the other columns alone
    torch.cuda.synchronize()
    assert torch.all(wide[:, 20:] == 7.0) and not torch.all(wide[:, :20] == 7.0)
    sim.close()


@pytest.mark.parametrize("n", [4096, 131072])
def test_batch_scale_parity_against_c_oracle(pkg, n):
    """The CUDA step against the float64 C oracle (oracle/quadx_oracle.c, pinned to the numpy oracle at 1e-9) at
    BASELINE.json's batch sizes -- configs[1] (4 096 envs) and the per-GPU shard of configs[3] / [4] (131 072 envs) -- with
    motor noise, auto-reset and the reference's reset protocol, 48 steps (every env passes the floor rule of step 32 or
    flies on).  An env whose termination falls on the other side of fp32 rounding (dome radius, floor threshold) is out of
    step from there on: such envs are dropped and their number is bounded; everything else must agree at every step.
    Rewards are compared on ALL remaining envs: where a camera pixel count flips (hover.py:209-213) the reward moves by up to
    one pixel's worth, those samples are counted against a stated rate instead of being skipped silently."""
    from oracle.c_oracle import COracle

    cfg = pkg.default_config()
    sim = pkg.QuadXSim(n, cfg, seed=31)
    orc = COracle(n, seed=31, auto_reset=True, noise=True)
    b = _Bufs(sim)
    sim.reset(b.obs)
    o2 = orc.reset().copy()
    _close(b.obs.cpu().numpy(), o2, 2e-3, "reset obs")
    rng = np.random.default_rng(5)
    acc = ForkAccount(n)
    lift = rng.uniform(0, 1, n) < 0.7  # 70 % of the fleet lifts off, the rest idles into the floor rule of step 32
    for k in range(48):
        a = rng.uniform(-1, 1, (n, 4)).astype(np.float32)
        a[:, :3] *= 0.2
        a[:, 3] = np.where(lift, 0.2 + 0.1 * a[:, 3], -0.9)
        o, r, te, tr = b.step(sim, a)
        o2, r2, te2, tr2, _ = orc.step(a.astype(np.float64))
        acc.step(o, r, te, tr, o2, r2, te2, tr2)
    print(f"n={n}: out-of-step envs {acc.out_of_step} (of which forked at a discontinuity: {acc.forked}), pixel-count flips {acc.flips}/{acc.seen}, "
          f"worst obs err {acc.worst_obs:.2e}, worst reward err {acc.worst_rew:.2e}")
    acc.check(max(4, n // 500))
    s1, s2 = sim.episode_stats(), orc.stats()
    assert abs(s1[2] - s2[2]) <= max(4, n // 500) and abs(s1[1] - s2[1]) <= 48 * max(4, n // 500)
    sim.close()


def test_raster_vision_mode_equals_reference_detector(pkg):
    """vision_mode = 1 (csrc/qx_model.cuh:vision_raster, H4): the camera columns of the observation against the reference's real
    detect_rectangle (hover.py:157-222) run on rasterised frames of the same poses (random in-dome poses put in through
    qx_set_state; the comparison is feature extraction only): visibility identical,
    contour area and bounding-box ratio the detector's own numbers (a boundary pixel may differ in fp32: counted), centre
    within 0.8 px, and the target term of the reward (hover.py:296-317) within 2e-2 -- against 0.45 for the analytic mode."""
    from oracle import vision
    from oracle.hover_oracle import detect_rectangle
    from oracle.quadx_model import QuadXParams

    n = 512
    cfg = pkg.default_config()
    # aviary_steps_per_step = 0: a step runs no physics, so the observation is built from exactly the pose that was set
    cfg.update(start_pos=[0, 0, 1.2], reset_idle_steps=0, auto_reset=0, noise=0, vision_mode=1, aviary_steps_per_step=0, max_steps=10000)
    rng = np.random.default_rng(3)
    p = QuadXParams()
    sim = pkg.QuadXSim(n, cfg, seed=78)
    b = _Bufs(sim)
    sim.reset(b.obs)
    st = sim.get_state()
    from oracle.quadx_model import euler_to_quat

    pos = rng.uniform(-1.8, 1.8, (n, 3)); pos[:, 2] = rng.uniform(0.3, 2.4, n)
    quat = euler_to_quat(rng.uniform(-0.4, 0.4, (n, 3)))
    for j, key in enumerate(("px", "py", "pz")):
        st[key] = pos[:, j].astype(np.float32)
    for j, key in enumerate(("qx", "qy", "qz", "qw")):
        st[key] = quat[:, j].astype(np.float32)
    sim.set_state(st)
    a = np.zeros((n, 4), np.float32)
    o, r, te, tr = b.step(sim, a)
    st2 = sim.get_state()
    pos2 = np.stack([st2["px"], st2["py"], st2["pz"]], 1).astype(np.float64)
    quat2 = np.stack([st2["qx"], st2["qy"], st2["qz"], st2["qw"]], 1).astype(np.float64)
    assert np.array_equal(pos2.astype(np.float32), pos.astype(np.float32))
    V, C, A, R = np.zeros(n, bool), np.zeros((n, 2)), np.zeros(n), np.zeros(n)
    for i in range(n):
        V[i], C[i], A[i], R[i] = detect_rectangle(vision.render_rgba(pos2[i], quat2[i], p))
    vis = o[:, 13] > 0.5
    vis_mis = int((vis != V).sum())
    both = vis & V
    assert both.sum() > 250 and vis_mis <= max(2, n // 100), (int(both.sum()), vis_mis)
    area_flip = np.abs(o[:, 11] - A)[both] > 1e-7
    ratio_flip = np.abs(o[:, 14] - R)[both] > 1e-6
    print(f"raster mode vs the reference detector: {int(both.sum())} frames, visibility mismatches {vis_mis}, area differs in {int(area_flip.sum())}, "
          f"ratio differs in {int(ratio_flip.sum())}, worst centre error {np.abs(o[:, 7:9] - C)[both].max() * 64:.2f} px")
    assert area_flip.sum() <= max(3, n // 50) and ratio_flip.sum() <= max(3, n // 50)  # a border pixel decided differently by the moved pose / fp32
    assert np.abs(o[:, 11] - A)[both].max() * 128 * 128 <= 3.0
    assert np.abs(o[:, 7:9] - C)[both].max() * 64 <= 1.0
    ok = both.copy(); ok[both] = ~(area_flip | ratio_flip)
    rew = lambda cc, aa, rr: -(np.hypot(cc[:, 0], cc[:, 1]) + np.abs(aa - 0.013) + np.abs(rr - 1.53))  # noqa: E731
    assert np.abs(rew(o[:, 7:9], o[:, 11], o[:, 14]) - rew(C, A, R))[ok].max() <= 2e-2
    sim.close()
