"""Shared helpers for the parity tests (oracle <-> CUDA state conversion)."""
import numpy as np


def oracle_to_kernel_state(orc) -> dict:
    """HoverVecOracle -> dict keyed like fpv_drone_rl_agent_b200.STATE_FIELDS."""
    from oracle.quadx_model import quat_to_mat

    st = orc.st
    wb = np.einsum("nji,nj->ni", quat_to_mat(st.quat), st.omega)  # the kernel carries body rates
    flags = (
        st.contact.astype(np.uint32) * 1
        | orc.terminated.astype(np.uint32) * 2
        | orc.truncated.astype(np.uint32) * 4
        | orc.info["out_of_bounds"].astype(np.uint32) * 8
        | orc.info["on_floor"].astype(np.uint32) * 16
        | (st.s_pos[:, 2] < orc.cfg.floor_threshold).astype(np.uint32) * 32
    )
    d = {
        "px": st.pos[:, 0], "py": st.pos[:, 1], "pz": st.pos[:, 2],
        "qx": st.quat[:, 0], "qy": st.quat[:, 1], "qz": st.quat[:, 2], "qw": st.quat[:, 3],
        "vx": st.vel[:, 0], "vy": st.vel[:, 1], "vz": st.vel[:, 2],
        "wbx": wb[:, 0], "wby": wb[:, 1], "wbz": wb[:, 2],
        "step_count": orc.step_count, "rng_ctr": orc.rng_ctr, "ep_return": orc.ep_return, "flags": flags,
        "prev_cx": orc.prev_centre[:, 0], "prev_cy": orc.prev_centre[:, 1], "prev_area": orc.prev_area, "prev_ratio": orc.prev_ratio,
        "prev_roll": orc.prev_euler[:, 0], "prev_pitch": orc.prev_euler[:, 1], "prev_yaw": orc.prev_euler[:, 2],
    }
    for m in range(4):
        d[f"thr{m}"] = st.thr[:, m]
        d[f"prev_a{m}"] = orc.prev_action[:, m]
    for a in range(3):
        d[f"pid_i{a}"] = st.pid_i[:, a]
        d[f"pid_e{a}"] = st.pid_e[:, a]
        d[f"s_wb{a}"] = st.s_wb[:, a]
        d[f"s_vb{a}"] = st.s_vb[:, a]
    return d


def kernel_state_arrays(s: dict):
    """-> pos[N,3], quat[N,4], vel[N,3], omega[N,3], thr[N,4]."""
    pos = np.stack([s["px"], s["py"], s["pz"]], 1)
    quat = np.stack([s["qx"], s["qy"], s["qz"], s["qw"]], 1)
    vel = np.stack([s["vx"], s["vy"], s["vz"]], 1)
    from oracle.quadx_model import quat_to_mat

    wb = np.stack([s["wbx"], s["wby"], s["wbz"]], 1).astype(np.float64)
    omega = np.einsum("nij,nj->ni", quat_to_mat(quat.astype(np.float64)), wb)  # world frame, like the oracle
    thr = np.stack([s[f"thr{m}"] for m in range(4)], 1)
    return pos, quat, vel, omega, thr


# obs columns produced by the camera (hover.py:257-263)
VISION_COLS = [7, 8, 9, 10, 11, 12, 13, 14, 15]
NONVISION_COLS = [0, 1, 2, 3, 4, 5, 6, 16, 17, 18, 19]


class ForkAccount:
    """Which envs of a CUDA hover sim are still in step with the float64 oracle, over a run of auto-reset steps.

    An env whose termination falls on the other side of fp32 rounding (dome radius, floor threshold) is out of step from there
    on, and so is one that takes a discontinuity of the model (floor plane touched one sub-step earlier, motor saturation on /
    off) on a different side than float64: its observations or reward jump apart.  Such envs are dropped from every later
    comparison and counted (`forked` of them at a discontinuity); the caller bounds the count.  Rewards are compared on every
    remaining env: where a camera pixel count flips (hover.py:209-213) the reward moves by up to one pixel's worth, and those
    samples are counted (`flips` of `seen`) instead of skipped.  `step` returns the envs still in step."""

    def __init__(self, n: int, obs_tol: float = 3e-3, rew_tol: float = 5e-3):
        self.sync = np.ones(n, bool)
        self.obs_tol, self.rew_tol = obs_tol, rew_tol
        self.forked = self.flips = self.seen = 0
        self.worst_obs = self.worst_rew = 0.0

    def step(self, o, r, te, tr, o2, r2, te2, tr2, also_fork=None) -> np.ndarray:
        """also_fork [n] bool: envs the caller found apart by a check of its own (e.g. of the terminal observation)."""
        self.sync &= (te == te2) & (tr == tr2)
        err = np.abs(o[:, NONVISION_COLS] - o2[:, NONVISION_COLS]).max(axis=1)
        same_px = (o[:, 13] == o2[:, 13]) & (np.abs(o[:, 14] - o2[:, 14]) < 1e-4)
        # (the yaw body rate enters the reward, hover.py:322-324, but not the observation: a fork can show there first)
        fork = self.sync & ((err > self.obs_tol) | (same_px & (np.abs(r - r2) > self.rew_tol)))
        if also_fork is not None:
            fork |= self.sync & also_fork
        self.forked += int(fork.sum())
        self.sync &= ~fork
        m = self.sync.copy()
        if m.any():
            self.worst_obs = max(self.worst_obs, float(err[m].max()))
        same = m & same_px
        self.flips += int((m & ~same).sum())
        self.seen += int(m.sum())
        if same.any():
            self.worst_rew = max(self.worst_rew, float(np.abs(r[same] - r2[same]).max()))
        # the flipped samples are not skipped: their reward error is bounded by one pixel row of the bbox ratio + visibility (0.45)
        if (m & ~same).any():
            assert float(np.abs(r[m & ~same] - r2[m & ~same]).max()) <= 2.5
        return m

    @property
    def out_of_step(self) -> int:
        return int((~self.sync).sum())

    def check(self, bound: int) -> None:
        assert self.out_of_step <= bound, (self.out_of_step, bound)
        assert self.flips <= 0.01 * self.seen, (self.flips, self.seen)
        assert self.worst_obs <= self.obs_tol and self.worst_rew <= self.rew_tol, (self.worst_obs, self.worst_rew)


class _DevWords:
    """int32 words at a raw device address, for torch.as_tensor (the CUDA array interface)."""

    def __init__(self, addr: int, n: int):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (addr, False), "version": 3}


def read_done_queue(sim) -> tuple[int, np.ndarray]:
    """(published count, the env indices it covers) of qx_done_queue, after a device synchronise."""
    import torch

    cnt, idx = sim.done_queue()
    torch.cuda.synchronize(sim.device)
    count = int(torch.as_tensor(_DevWords(cnt.value, 1), device=sim.device).cpu()[0])
    assert 0 <= count <= sim.n, count
    return count, torch.as_tensor(_DevWords(idx.value, sim.n), device=sim.device)[:count].cpu().numpy()


def check_done_queue(sim, done: np.ndarray) -> tuple[int, np.ndarray]:
    """The queue of the step just begun holds every finished env once and nothing else."""
    count, idx = read_done_queue(sim)
    want = np.flatnonzero(done)
    assert count == want.size, (count, want.size)
    assert np.array_equal(np.sort(idx), want), "done queue: wrong or duplicated env indices"
    return count, idx


# PyFlyt flight modes (-1..7): how a Box(-1, 1) action is scaled into each mode's setpoint in the tests
# (action_scale for the first three channels, thrust_scale * a3 + thrust_bias for the fourth)
FLIGHT_MODE_SCALING = {
    -1: dict(action_scale=(0.0, 0.0, 0.0), thrust_scale=0.0003, thrust_bias=0.53),  # four motor pwm, all via thrust_scale / bias (open loop: keep it gentle)
    0: dict(action_scale=(30.0, 30.0, -30.0), thrust_scale=0.5, thrust_bias=0.5),  # hover.py:337-341
    1: dict(action_scale=(0.3, 0.3, 1.0), thrust_scale=1.0, thrust_bias=0.0),      # p, q, r [rad], vz [m/s]
    2: dict(action_scale=(0.3, 0.3, 1.0), thrust_scale=0.5, thrust_bias=1.2),      # vp, vq, vr [rad/s], z [m]
    3: dict(action_scale=(0.3, 0.3, 1.0), thrust_scale=0.5, thrust_bias=1.2),      # p, q, r, z
    4: dict(action_scale=(1.0, 1.0, 1.0), thrust_scale=0.5, thrust_bias=1.2),      # u, v [m/s], vr, z
    5: dict(action_scale=(1.0, 1.0, 1.0), thrust_scale=1.0, thrust_bias=0.0),      # u, v, vr, vz
    6: dict(action_scale=(1.0, 1.0, 1.0), thrust_scale=1.0, thrust_bias=0.0),      # vx, vy, vr, vz
    7: dict(action_scale=(1.0, 1.0, 1.5), thrust_scale=0.5, thrust_bias=1.2),      # x, y [m], r [rad], z
}
