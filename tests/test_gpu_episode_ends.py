"""GPU: what happens when an episode ends on the large-batch env step -- the lean hot kernel and the reset queue that
qx_create selects from 32 768 envs up, driven the way the PPO rollout drives it (qx_step_begin, read the done queue and
the terminal observations, qx_step_end).

  * whole episodes against the float64 C oracle at training sizes, ending every way an episode ends (time limit, dome
    exit, floor rule), with terminal observations, next-episode observations and the Monitor sums checked at every step;
  * the done queue (qx_done_queue) exactly, from all three code paths that publish it;
  * the speculative floor re-run of the paired hot kernel (hot_substeps_spec), entered by construction;
  * the yaw task through the reset queue;
  * misaligned step buffers are refused before anything is launched, aligned column views are accepted.

Tolerances are those of tests/test_gpu_parity.py (test_batch_scale_parity_against_c_oracle, with its fork accounting in
tests/util.py:ForkAccount, and test_state_roundtrip_and_oracle_injection) and tests/test_yaw.py.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from tests.util import NONVISION_COLS, ForkAccount, check_done_queue, kernel_state_arrays, oracle_to_kernel_state, read_done_queue

pytestmark = pytest.mark.gpu

HOVER_THR = float(np.sqrt(0.1 * 9.81 / 4.0))  # pwm at which thrust = weight (cf2x.yaml:2, cf2x.urdf:10)
CAM_COLS = [7, 8, 9, 10, 11, 12]  # centre, previous centre, area, previous area (hover.py:253-267)
TUNING_VARS = ("QX_HOT", "QX_LANES", "QX_SHAPE", "QX_MERGED", "QX_PAIRED_RESET", "QX_STREAM_STORES", "QX_PDL", "QX_FORCE_GENERIC")
F_CONTACT, F_OOB, F_ONFLOOR = 1, 8, 16  # flags-word bits (qx_get_flags)
QX_EINVAL = -1

# the large-batch selections stepped in lockstep with one oracle: the default (hot kernel, paired lanes, two launches),
# the generic kernels, and the merged launch
HANDLES = {"default": {}, "generic": {"QX_HOT": "0"}, "merged": {"QX_MERGED": "1"}}


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge

    ge.build()
    import fpv_drone_rl_agent_b200 as pkg

    return pkg


def _sim(pkg, monkeypatch, env, n, cfg, seed, **kw):
    """A QuadXSim created under exactly the QX_* variables in `env` (they are read at qx_create)."""
    for k in TUNING_VARS:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    return pkg.QuadXSim(n, cfg, seed=seed, **kw)


class _Stepper:
    """One handle and its output buffers, stepped as the rollout steps it: step_begin, the done queue (checked), the flags
    words before the reset (reasons), step_end, the queue again (still readable while / after the reset runs)."""

    def __init__(self, sim):
        n, d, od = sim.n, sim.device, sim.obs_dim
        self.sim = sim
        self.obs = torch.zeros(n, od, device=d)
        self.rew = torch.zeros(n, device=d)
        self.te = torch.zeros(n, dtype=torch.uint8, device=d)
        self.tr = torch.zeros(n, dtype=torch.uint8, device=d)
        self.tobs = torch.zeros(n, od, device=d)
        self.queue_lengths = set()
        self.tally = _Tally(n)  # the Monitor sums of the returned flags and rewards: qx_episode_stats must say the same

    def step(self, a: torch.Tensor, want_flags: bool = False):
        self.sim.step_begin(a, self.obs, self.rew, self.te, self.tr, self.tobs)
        torch.cuda.synchronize(self.sim.device)
        te, tr = self.te.cpu().numpy().astype(bool), self.tr.cpu().numpy().astype(bool)
        done = te | tr
        count, idx = check_done_queue(self.sim, done)
        flags = self.sim.flags() if want_flags else None  # the finished envs' words still hold the end reason until step_end
        self.sim.step_end(self.obs)
        count2, idx2 = read_done_queue(self.sim)
        assert count2 == count and np.array_equal(idx2, idx), "the done queue changed under step_end"
        self.queue_lengths.add(count)
        o, r, t = self.obs.cpu().numpy(), self.rew.cpu().numpy(), self.tobs.cpu().numpy()
        self.tally.add(r, done)
        return o, r, te, tr, t, flags

    def check_stats(self):
        s, l, c = self.sim.episode_stats()
        self.tally.check(s, l, c)
        return s, l, c


class _Tally:
    """SB3 Monitor's sums (return, length, count of the finished episodes) kept from a sim's per-step rewards and flags."""

    def __init__(self, n):
        self.ep_ret, self.ep_len = np.zeros(n), np.zeros(n, np.int64)
        self.sum_ret, self.sum_len, self.n_done = 0.0, 0, 0
        self.episodes = np.zeros(n, np.int64)  # per env

    def add(self, r, done):
        self.ep_ret += r
        self.ep_len += 1
        self.sum_ret += float(self.ep_ret[done].sum())
        self.sum_len += int(self.ep_len[done].sum())
        self.n_done += int(done.sum())
        self.episodes += done
        self.ep_ret[done], self.ep_len[done] = 0.0, 0

    def check(self, s, l, c):
        assert (c, l) == (self.n_done, self.sum_len), ((c, l), (self.n_done, self.sum_len))
        assert abs(s - self.sum_ret) <= 1e-4 * max(1.0, abs(self.sum_ret)), (s, self.sum_ret)


def _aviary_state(orc) -> np.ndarray:
    """[N,4,3] rows (body rates, Euler, body velocity, position) of the C oracle's state, for oracle.test_policy."""
    from oracle.quadx_model import quat_to_euler, quat_to_mat

    s = orc.state()
    pos, quat, vel, om = s[:, 0:3], s[:, 3:7], s[:, 7:10], s[:, 10:13]
    R = quat_to_mat(quat)
    return np.stack([np.einsum("nji,nj->ni", R, om), quat_to_euler(quat), np.einsum("nji,nj->ni", R, vel), pos], axis=1)


# (n, max_steps, steps run, out-of-step envs measured on a B200 -- the same on all three handles, which agree bit for bit).
# The bound is three times the measured count: forks are envs that sit within fp32 rounding of a discontinuity, a property
# of the seeded trajectories, so a kernel that changes what it computes shows up as many more.
EPISODE_RUNS = [(32768, 60, 130, 13), (131072, 60, 130, 34), (32768, 400, 404, 109)]
FORK_BOUND_FACTOR = 3


@pytest.mark.parametrize("n,max_steps,steps,forks_measured", EPISODE_RUNS)
def test_episode_ends_against_c_oracle(pkg, monkeypatch, n, max_steps, steps, forks_measured):
    """Whole episodes of the default config (floor spawn, 10 idle steps, motor noise, auto-reset) on the three large-batch
    selections against the float64 C oracle.  A third of the envs hover under the test policy into the time limit, a third
    climb tilted out of the flight dome, a third idle into the floor rule of step 32: every end happens many times, on
    different steps in one warp.  At every step, on the envs in step with the oracle: flags exact, reward and observation
    (for a finished env: the first one of its next episode) within the scale test's bounds, the terminal observation of
    every finished env against the oracle's, the done queue exactly; at the end qx_episode_stats against the flags."""
    from oracle.c_oracle import COracle
    from oracle.test_policy import hover_actions

    cfg = pkg.default_config()
    cfg.update(max_steps=max_steps, auto_reset=1)
    steppers = {name: _Stepper(_sim(pkg, monkeypatch, env, n, cfg, seed=31)) for name, env in HANDLES.items()}
    for s in steppers.values():
        assert s.sim.lib.qx_uses_reference_constants(s.sim._h) == 1  # max_steps is not a model constant
    orc = COracle(n, seed=31, auto_reset=True, noise=True, max_steps=max_steps)
    o2 = orc.reset().copy()
    for s in steppers.values():
        s.sim.reset(s.obs)
        torch.cuda.synchronize()
        assert np.abs(s.obs.cpu().numpy()[:, NONVISION_COLS] - o2[:, NONVISION_COLS]).max() <= 2e-3
    group = np.arange(n) % 3  # 0: hover into the time limit, 1: climb out of the dome, 2: zero thrust into the floor rule
    rng = np.random.default_rng(7)
    tgt = np.stack([rng.uniform(-0.5, 0.5, n), rng.uniform(-0.5, 0.5, n), rng.uniform(0.8, 1.5, n)], 1)
    tilt = rng.uniform(-0.03, 0.03, (n, 2))
    accs = {name: ForkAccount(n) for name in steppers}
    t_flips = {name: 0 for name in steppers}
    t_seen = {name: 0 for name in steppers}
    t_worst = {name: 0.0 for name in steppers}
    reasons = {"time limit": 0, "dome": 0, "floor": 0}
    orc_tally = _Tally(n)
    d = steppers["default"].sim.device
    for k in range(steps):
        a = np.zeros((n, 4))
        a[group == 0] = hover_actions(_aviary_state(orc), tgt)[group == 0]
        a[group == 1, :2] = tilt[group == 1]
        a[group == 1, 3] = 1.0
        a[group == 2, 3] = -1.0
        a = a.astype(np.float32)
        a_dev = torch.from_numpy(a).to(d)
        outs = {name: s.step(a_dev, want_flags=name == "default") for name, s in steppers.items()}
        o2, r2, te2, tr2, info = orc.step(a.astype(np.float64))
        t2 = info["terminal_obs"]
        orc_tally.add(r2, te2 | tr2)
        for name, (o, r, te, tr, t, flags) in outs.items():
            done = (te | tr) & (te2 | tr2)
            # terminal observation: non-camera columns 2e-3; camera columns where the pixel counts agree (hover.py:209-213)
            terr = np.zeros(n)
            terr[done] = np.abs(t[done][:, NONVISION_COLS] - t2[done][:, NONVISION_COLS]).max(1)
            tsame = done & (t[:, 13] == t2[:, 13]) & (np.abs(t[:, 14] - t2[:, 14]) < 1e-4)
            terr[tsame] = np.maximum(terr[tsame], np.abs(t[tsame][:, CAM_COLS] - t2[tsame][:, CAM_COLS]).max(1))
            m = accs[name].step(o, r, te, tr, o2, r2, te2, tr2, also_fork=terr > 2e-3)
            md = m & done
            if md.any():
                t_worst[name] = max(t_worst[name], float(terr[md].max()))
            t_seen[name] += int(md.sum())
            t_flips[name] += int((md & ~tsame).sum())
            if flags is not None:
                reasons["time limit"] += int((md & tr).sum())
                reasons["dome"] += int((md & te & (flags & F_OOB != 0)).sum())
                reasons["floor"] += int((md & te & (flags & F_ONFLOOR != 0)).sum())
    bound = FORK_BOUND_FACTOR * forks_measured
    orc_tally.check(*orc.stats())
    for name, s in steppers.items():
        acc = accs[name]
        print(f"n={n} max_steps={max_steps} [{name}]: out-of-step envs {acc.out_of_step} (forked at a discontinuity {acc.forked}, "
              f"measured once {forks_measured}, bound {bound}), pixel-count flips {acc.flips}/{acc.seen}, terminal obs: {t_seen[name]} compared, {t_flips[name]} "
              f"pixel-count flips, worst err {t_worst[name]:.2e}; worst obs err {acc.worst_obs:.2e}, worst reward err {acc.worst_rew:.2e}; "
              f"queue lengths seen: {len(s.queue_lengths)} distinct, max {max(s.queue_lengths)}")
        acc.check(bound)
        assert t_flips[name] <= 0.01 * max(1, t_seen[name]), (t_flips[name], t_seen[name])
        s.check_stats()
        # qx_episode_stats follows the flags, the oracle's Monitor sums follow its flags, and the envs in step end their episodes
        # on the same steps: the two sums differ by what the out-of-step envs contribute, nothing else
        assert np.array_equal(s.tally.episodes[acc.sync], orc_tally.episodes[acc.sync])
        assert 0 in s.queue_lengths and len(s.queue_lengths) > 3
        s.sim.close()
    print(f"n={n} max_steps={max_steps}: ends by reason (envs in step, default handle): {reasons}")
    assert reasons["time limit"] >= n // 10 and reasons["dome"] >= n // 10 and reasons["floor"] >= n // 10, reasons


@pytest.mark.parametrize("env", [{}, {"QX_HOT": "0"}, {"QX_MERGED": "1"}, {"QX_LANES": "1"}, {"QX_PAIRED_RESET": "0"},
                                 {"QX_PAIRED_RESET": "0", "QX_MERGED": "1"}], ids=lambda e: ",".join(f"{k}={v}" for k, v in e.items()) or "default")
def test_done_queue_mass_end_and_quiet_steps(pkg, monkeypatch, env):
    """Zero thrust from the floor: nothing ends for 31 steps, then every env on its 32nd (the floor rule), then nothing again.
    The queue is exact on every step, from each of its producers: the generic deferred kernel, the two-launch hot kernel and
    the merged launch's exit ticket."""
    n = 32768 + 77
    cfg = pkg.default_config()
    cfg.update(auto_reset=1)
    s = _Stepper(_sim(pkg, monkeypatch, env, n, cfg, seed=2))
    s.sim.reset(s.obs)
    a = torch.zeros(n, 4, device=s.sim.device)
    a[:, 3] = -1.0
    ends = []
    for k in range(36):
        _, _, te, tr, _, _ = s.step(a)
        if (te | tr).any():
            ends.append((k, int((te | tr).sum())))
    assert ends == [(31, n)], ends
    assert s.queue_lengths == {0, n}
    s.check_stats()
    s.sim.close()


def _spec_scene(n_warps_full=4, tail=13, seed=3):
    """HoverVecOracle states laid out in warps of 32 envs (the paired hot kernel runs one env per thread):
      warp 0: every env inverted near the floor ("dive");   warp 1: one dive at lane 7, the rest hovering at 1 m;
      warp 2: one env resting on the floor (contact: the warp takes the full loop) and dives at lanes 1-8;
      warp 3: all hovering;   tail: `tail` envs (a ragged warp), dives at the even lanes.
    A dive: rolled 155-166 deg (upside down, clear of the +-pi ambiguity of Euler angles), motors at full throttle and thrust
    command 1 with zero rate commands (about 4.7 g downwards), 5 steps into the episode (inside the floor rule's grace),
    started 50-60 mm up at 0-0.1 m/s down -- high enough that the predictor of hot_substeps_spec clears it by more than
    5 mm, low enough that the drone reaches the floor within the agent step (it drops about 58 mm in 0.05 s)."""
    from oracle.hover_oracle import HoverConfig, HoverVecOracle
    from oracle.quadx_model import QuadXParams, euler_to_quat, take_snapshot

    n = 32 * n_warps_full + tail
    orc = HoverVecOracle(n, QuadXParams(), HoverConfig(start_pos=(0, 0, 1.0), spawn_throttle=HOVER_THR, reset_idle_steps=0), seed=seed, noise=True)
    orc.reset()
    rng = np.random.default_rng(seed)
    dive = np.zeros(n, bool)
    dive[0:32] = True
    dive[32 + 7] = True
    dive[64 + 1:64 + 9] = True
    dive[128::2] = True
    rest = np.zeros(n, bool)
    rest[64] = True
    st = orc.st
    nd = int(dive.sum())
    st.pos[dive] = np.stack([rng.uniform(-0.2, 0.2, nd), rng.uniform(-0.2, 0.2, nd), rng.uniform(0.05, 0.06, nd)], 1)
    st.quat[dive] = euler_to_quat(np.stack([rng.uniform(2.7, 2.9, nd), np.zeros(nd), rng.uniform(-0.5, 0.5, nd)], 1))
    st.vel[dive] = np.stack([np.zeros(nd), np.zeros(nd), rng.uniform(-0.1, 0.0, nd)], 1)
    st.omega[dive] = 0.0
    st.thr[dive] = 1.0
    st.pos[rest] = np.array([0.0, 0.0, orc.p.floor_z])
    st.vel[rest] = st.omega[rest] = 0.0
    st.thr[rest] = orc.p.pwm_idle
    for m in (dive, rest):
        st.pid_i[m] = st.pid_e[m] = 0.0
        st.contact[m] = False
    st.contact[rest] = True
    take_snapshot(st)
    orc.prev_euler = st.s_euler.copy()
    orc.step_count[:] = 5
    a = np.zeros((n, 4))
    a[:, 3] = 2 * HOVER_THR - 1
    a[dive, 3] = 1.0
    a[rest, 3] = -1.0
    return orc, dive, rest, a


def _predictor_clears(cfg, pz, vz, contact, margin):
    """float32 restatement of hot_substeps_spec's predictor: pz + min(vz, 0) T - g T^2 > floor_z (+ margin), T = n_sub_step h."""
    f = np.float32
    h = f(1.0 / cfg.physics_hz)
    T = f(f(cfg.aviary_steps_per_step * int(cfg.physics_hz / cfg.control_hz)) * h)
    reach = f(np.minimum(vz.astype(f), f(0)).astype(np.float64) * T + pz.astype(f)) - f(f(f(cfg.gravity) * T) * T)
    return ~contact & (reach > f(cfg.floor_z) + f(margin))


def test_speculative_floor_rerun(pkg, monkeypatch):
    """hot_substeps_spec runs a warp that no env of it is predicted to bring near the floor without the floor stand-in, and
    re-runs the full loop for an env whose lowest pz still went below floor_z.  Envs built to take that branch must end the
    step resting on the floor (pz == floor_z, contact flag set: the speculative result has neither), bit for bit what the
    generic kernel computes, merged or not, and within the one-step bounds of the float64 oracle."""
    orc, dive, rest, a = _spec_scene()
    n = orc.n
    cfg = pkg.default_config()
    cfg.update(start_pos=[0, 0, 1.0], spawn_throttle=HOVER_THR, reset_idle_steps=0, auto_reset=1)
    ks = oracle_to_kernel_state(orc)
    # the scene is what it claims: every dive clears the predictor by >= 5 mm, and warp 2 is made slow by its resting env
    clears = _predictor_clears(cfg, ks["pz"].astype(np.float32), ks["vz"].astype(np.float32), (ks["flags"] & F_CONTACT) != 0, 0.005)
    assert clears[dive].all() and not clears[rest].any()
    warp = np.arange(n) // 32
    slow_warp = np.array([not clears[warp == w].all() for w in range(warp.max() + 1)])
    rerun = dive & ~slow_warp[warp]  # dives the speculative loop runs first
    outs = []
    for env in ({"QX_HOT": "0"}, {"QX_HOT": "1", "QX_LANES": "4", "QX_MERGED": "0"}, {"QX_HOT": "1", "QX_LANES": "4", "QX_MERGED": "1"}):
        sim = _sim(pkg, monkeypatch, env, n, cfg, seed=3)
        s = _Stepper(sim)
        sim.reset(s.obs)
        sim.set_state(ks)
        o, r, te, tr, t, flags = s.step(torch.as_tensor(a, dtype=torch.float32, device=sim.device), want_flags=True)
        outs.append((env, o, r, te, tr, flags, sim.get_state()))
        sim.close()
    o2, r2, te2, tr2, _ = orc.step(a)
    _, o1, r1, te1, tr1, f1, s1 = outs[0]
    assert not (te1 | tr1).any()
    for env, o, r, te, tr, flags, st in outs:
        assert np.all(st["pz"][dive] == np.float32(cfg.floor_z)) and np.all(flags[dive] & F_CONTACT), env
        assert np.array_equal(o.view(np.uint32), o1.view(np.uint32)) and np.array_equal(r.view(np.uint32), r1.view(np.uint32)), env
        assert np.array_equal(te, te1) and np.array_equal(tr, tr1) and np.array_equal(flags, f1), env
        for key in st:
            assert np.array_equal(st[key].view(np.uint32), s1[key].view(np.uint32)), (env, key)
    # against the oracle (test_gpu_parity.py:test_state_roundtrip_and_oracle_injection's one-step bounds)
    assert np.array_equal(te1, te2) and np.array_equal(tr1, tr2) and np.array_equal(orc.st.contact, (f1 & F_CONTACT) != 0)
    pos, quat, vel, om, thr = kernel_state_arrays(s1)
    for x, y, tol, what in ((pos, orc.st.pos, 2e-6, "pos"), (vel, orc.st.vel, 2e-5, "vel"), (om, orc.st.omega, 2e-4, "omega"), (thr, orc.st.thr, 1e-5, "thr")):
        err = np.abs(x - y) / np.maximum(1.0, np.abs(y))
        assert err.max() <= tol, (what, float(err.max()))
    same = (o1[:, 13] == o2[:, 13]) & (np.abs(o1[:, 14] - o2[:, 14]) < 1e-4)
    assert np.abs(o1[:, NONVISION_COLS] - o2[:, NONVISION_COLS]).max() <= 2e-3 and np.abs(r1[same] - r2[same]).max() <= 2e-3
    print(f"speculative floor re-run: {int(rerun.sum())} envs took the re-run branch ({int(dive.sum())} dives, "
          f"{int((dive & ~rerun).sum())} of them in a warp made slow by a resting env); all landed on the floor")
    assert rerun.sum() >= 32 + 1 + 7


def test_yaw_through_reset_queue(pkg, monkeypatch):
    """The yaw task above the inline-reset limit (16 384 envs): its finished envs go through the generic deferred kernel and
    the reset-queue launch.  Two episodes against the oracle under test_yaw.py's bounds, terminal observations included,
    and the done queue exactly."""
    from oracle.yaw_oracle import YawConfig, YawVecOracle

    n, max_steps = 20000, 24
    cfg = pkg.default_config(pkg.QX_TASK_YAW)
    cfg.update(max_steps=max_steps, cam_tilt_up_deg=20.0, auto_reset=1)  # a camera that sees the sphere (test_yaw.py)
    s = _Stepper(_sim(pkg, monkeypatch, {}, n, cfg, seed=4, task=pkg.QX_TASK_YAW))
    orc = YawVecOracle(n, cfg=YawConfig(cam_tilt_up_deg=20.0, max_steps=max_steps), seed=4, noise=True)
    s.sim.reset(s.obs)
    torch.cuda.synchronize()
    assert np.abs(s.obs.cpu().numpy() - orc.reset()).max() < 2e-3
    rng = np.random.default_rng(0)
    cols = [0, 1, 2, 5, 6, 7, 8, 9, 10, 11]

    def close(o, o2, r, r2, what):
        same = (o[:, 3] != 0) == (o2[:, 3] != 0)  # a sphere within fp32 rounding of the image border may flip visibility
        assert same.mean() > 0.995, what
        assert np.abs(o[:, cols] - o2[:, cols]).max() < 3e-3, (what, np.abs(o[:, cols] - o2[:, cols]).max())
        assert np.abs(o[same][:, 3:5] - o2[same][:, 3:5]).max(initial=0.0) < 2e-3, what
        if r is not None:
            assert np.abs(r[same] - r2[same]).max() < 3e-3, what

    ends = []
    for k in range(2 * (max_steps + 1) + 2):
        if k % 10 == 0:
            a = (0.3 * rng.uniform(-1, 1, n)).astype(np.float32)
        o, r, te, tr, t, _ = s.step(torch.as_tensor(a, device=s.sim.device).view(n, 1))
        o2, r2, te2, tr2, info = orc.step(a.astype(np.float64))
        assert np.array_equal(te, te2) and np.array_equal(tr, tr2), k
        close(o, o2, r, r2, f"obs @ {k}")
        done = te | tr
        if done.any():
            ends.append(k)
            close(t[done], info["terminal_obs"][done], None, None, f"terminal obs @ {k}")
            assert np.all(o[done][:, 8:12] == 0)  # the next episode starts with a cleared action history (yaw.py:90-92)
    assert ends == [max_steps, 2 * max_steps + 1], ends
    _, l, c = s.check_stats()
    assert c == 2 * n and l == 2 * (max_steps + 1) * n
    s.sim.close()


def _bufs(n, d, od=20):
    return (torch.zeros(n, device=d), torch.zeros(n, dtype=torch.uint8, device=d), torch.zeros(n, dtype=torch.uint8, device=d),
            torch.zeros(n, od, device=d))


def _offset(shape, elems, dtype=torch.float32, fill=7.0):
    """A contiguous tensor of `shape` that starts `elems` elements into its allocation (the allocation itself is aligned)."""
    flat = torch.full((int(np.prod(shape)) + elems,), fill, dtype=dtype, device="cuda")
    return flat[elems:].view(*shape), flat


@pytest.mark.parametrize("n", [1000, 32768])
def test_misaligned_step_buffers_are_refused(pkg, monkeypatch, n):
    """A buffer the kernels would access with a misaligned vector instruction is refused before anything is launched --
    ValueError naming it from the Python wrappers, QX_EINVAL from the C-ABI -- and nothing is written: observation views
    whose rows are written as 16-byte (f32) / 8-byte (bf16) vectors, hover actions (one float4 per env), terminal
    observations (float4 rows), for qx_reset, qx_step (both reset paths), qx_step_begin, qx_step_end and qx_step_k."""
    cfg = pkg.default_config()
    cfg.update(auto_reset=1)
    sim = _sim(pkg, monkeypatch, {}, n, cfg, seed=1)
    L, d = sim.lib, sim.device
    rew, te, tr, tobs = _bufs(n, d)
    obs = torch.zeros(n, 20, device=d)
    act = torch.zeros(n, 4, device=d)
    sim.reset(obs)
    sim.step(act, obs, rew, te, tr, tobs)
    torch.cuda.synchronize()
    state0 = sim.get_state()
    wide = torch.full((n, 24), 7.0, device=d)
    wide16 = torch.full((n, 24), 7.0, device=d, dtype=torch.bfloat16)
    bad_obs = {"f32 +8 B": wide[:, 2:22], "f32 +4 B": wide[:, 1:21], "bf16 +2 B": wide16[:, 1:21], "bf16 +4 B": wide16[:, 2:22]}
    bad_act, act_alloc = _offset((n, 4), 1, fill=0.0)
    bad_tobs, tobs_alloc = _offset((n, 20), 2)
    bad_k_act, k_act_alloc = _offset((2, n, 4), 2, fill=0.0)
    bad_k_obs, k_obs_alloc = _offset((2, n, 20), 1)
    k_rew, k_te, k_tr = torch.zeros(2, n, device=d), torch.zeros(2, n, dtype=torch.uint8, device=d), torch.zeros(2, n, dtype=torch.uint8, device=d)
    k_act, k_obs = torch.zeros(2, n, 4, device=d), torch.zeros(2, n, 20, device=d)
    launches = L.qx_launch_count()
    py_calls = []
    for what, v in bad_obs.items():
        py_calls += [("obs", lambda v=v: sim.reset(v)), ("obs", lambda v=v: sim.step(act, v, rew, te, tr, tobs)),
                     ("obs", lambda v=v: sim.step(act, v, rew, te, tr, tobs, split=True)),
                     ("obs", lambda v=v: sim.step_begin(act, v, rew, te, tr, tobs)), ("obs", lambda v=v: sim.step_end(v))]
    py_calls += [("actions", lambda: sim.step(bad_act, obs, rew, te, tr, tobs)), ("actions", lambda: sim.step_begin(bad_act, obs, rew, te, tr)),
                 ("terminal_obs", lambda: sim.step(act, obs, rew, te, tr, bad_tobs)),
                 ("terminal_obs", lambda: sim.step(act, obs, rew, te, tr, bad_tobs, split=True)),
                 ("terminal_obs", lambda: sim.step_begin(act, obs, rew, te, tr, bad_tobs)),
                 ("actions", lambda: sim.step_k(bad_k_act, k_obs, k_rew, k_te, k_tr)), ("obs", lambda: sim.step_k(k_act, bad_k_obs, k_rew, k_te, k_tr))]
    for name, call in py_calls:
        with pytest.raises(ValueError, match=name):
            call()
    # the same buffers straight through the C-ABI
    vp, s = C.c_void_p, pkg._lib.stream(d)
    p = lambda t: vp(t.data_ptr())  # noqa: E731
    c_calls = []
    for v in bad_obs.values():
        code = 1 if v.dtype == torch.bfloat16 else 0
        c_calls += [L.qx_reset(sim._h, None, p(v), code, 24, s),
                    L.qx_step(sim._h, p(act), p(v), code, 24, p(rew), p(te), p(tr), p(tobs), s),
                    L.qx_step_begin(sim._h, p(act), p(v), code, 24, p(rew), p(te), p(tr), p(tobs), s),
                    L.qx_step_end(sim._h, p(v), code, 24, s)]
    c_calls += [L.qx_step(sim._h, p(bad_act), p(obs), 0, 20, p(rew), p(te), p(tr), None, s),
                L.qx_step_begin(sim._h, p(bad_act), p(obs), 0, 20, p(rew), p(te), p(tr), None, s),
                L.qx_step(sim._h, p(act), p(obs), 0, 20, p(rew), p(te), p(tr), p(bad_tobs), s),
                L.qx_step_begin(sim._h, p(act), p(obs), 0, 20, p(rew), p(te), p(tr), p(bad_tobs), s),
                L.qx_step_k(sim._h, 2, p(bad_k_act), p(k_obs), p(k_rew), p(k_te), p(k_tr), s),
                L.qx_step_k(sim._h, 2, p(k_act), p(bad_k_obs), p(k_rew), p(k_te), p(k_tr), s)]
    assert c_calls == [QX_EINVAL] * len(c_calls), c_calls
    assert b"aligned" in L.qx_last_error()
    torch.cuda.synchronize()
    assert L.qx_launch_count() == launches  # nothing was launched
    for t in (wide, wide16, tobs_alloc[2:], k_obs_alloc[1:]):
        assert torch.all(t == 7.0)
    st = sim.get_state()
    for key in st:
        assert np.array_equal(st[key].view(np.uint32), state0[key].view(np.uint32)), key
    # an odd row stride is written element by element: any element offset is fine
    odd = torch.zeros(n, 21, device=d)
    assert L.qx_reset(sim._h, None, p(odd[:, 1:21]), 0, 21, s) == 0
    sim.close()


@pytest.mark.parametrize("n", [1000, 32768])
def test_aligned_column_views_equal_contiguous_run(pkg, monkeypatch, n):
    """Observation views that are aligned are accepted and give the contiguous buffer's results bit for bit, through resets
    (the floor rule of step 32): buf[:, 4:24] of [n, 24] in f32 and in bf16 (16- / 8-byte vector rows), and buf[:, 1:21] of
    [n, 21] (odd row stride: element stores).  The columns outside the view are never written."""
    cfg = pkg.default_config()
    cfg.update(auto_reset=1)
    g = torch.Generator(device="cuda").manual_seed(3)
    steps = 40
    acts = (torch.rand(steps, n, 4, device="cuda", generator=g) * 2 - 1) * torch.tensor([0.3, 0.3, 0.3, 1.0], device="cuda")
    acts[:, : n // 2, 3] = -1.0  # half the fleet stays on the floor and is reset on step 32
    layouts = {"f32": (torch.float32, 20, 0), "bf16": (torch.bfloat16, 20, 0), "f32 [4:24] of 24": (torch.float32, 24, 4),
               "bf16 [4:24] of 24": (torch.bfloat16, 24, 4), "f32 [1:21] of 21": (torch.float32, 21, 1)}
    res = {}
    for name, (dt, width, c0) in layouts.items():
        sim = _sim(pkg, monkeypatch, {}, n, cfg, seed=9)
        rew, te, tr, tobs = _bufs(n, sim.device)
        buf = torch.full((steps + 1, n, width), 7.0, device=sim.device, dtype=dt)
        sim.reset(buf[0][:, c0:c0 + 20])
        for k in range(steps):
            sim.step(acts[k], buf[k + 1][:, c0:c0 + 20], rew, te, tr, tobs)
        torch.cuda.synchronize()
        assert torch.all(buf[..., :c0] == 7.0) and torch.all(buf[..., c0 + 20:] == 7.0), name
        assert sim.episode_stats()[2] >= n // 2  # the floor rule ended episodes, and step_end wrote through the view
        res[name] = buf[..., c0:c0 + 20].clone()
        sim.close()
    assert torch.equal(res["f32"].view(torch.int32), res["f32 [4:24] of 24"].view(torch.int32))
    assert torch.equal(res["f32"].view(torch.int32), res["f32 [1:21] of 21"].view(torch.int32))
    assert torch.equal(res["bf16"].view(torch.int16), res["bf16 [4:24] of 24"].view(torch.int16))
    assert torch.equal(res["f32"].to(torch.bfloat16).view(torch.int16), res["bf16"].view(torch.int16))
