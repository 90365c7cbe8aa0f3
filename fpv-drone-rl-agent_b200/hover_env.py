"""Host-side mirror of the reference's env interface on top of libquadx_b200.so.

  * ``QuadXHoverVecEnv`` -- what ``train_hover.py:42-43`` consumes: an SB3-style
    ``VecEnv`` (``reset() -> obs[N,20]``, ``step_async`` / ``step_wait`` ->
    ``(obs, rew, done, infos)``, auto-reset with ``terminal_observation``,
    ``TimeLimit.truncated`` and Monitor's ``episode`` statistics), but batched on
    one GPU with tensors that never leave the device.
  * ``QuadXHoverEnv`` -- the ``gymnasium.Env``-shaped single-env facade with the
    reference's signatures (``hover.py:72,334,363``), spaces (``hover.py:61,70``)
    and ``info`` keys (``hover.py:53-57``).

gymnasium / stable-baselines3 are not imported: the classes are duck-typed so
that they work where those packages are absent (SURVEY 8b).
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import QX_FRAME_MASK, QX_FRAME_RGBA, QX_OBS_BF16, QX_OBS_F32, QX_STATE_WORDS, QX_STATE_WORDS_CASCADE, QX_TASK_HOVER, QxConfig, check, default_config, expect, ptr, stream

# names of the 44 carried state words, in plane order (see csrc/qx_model.cuh Env)
STATE_FIELDS = (
    "px py pz qx qy qz qw vx vy vz wbx wby wbz thr0 thr1 thr2 thr3 pid_i0 pid_i1 pid_i2 pid_e0 pid_e1 pid_e2 "
    "s_wb0 s_wb1 s_wb2 s_vb0 s_vb1 s_vb2 step_count rng_ctr flags prev_roll prev_pitch prev_yaw ep_return "
    "prev_a0 prev_a1 prev_a2 prev_a3 prev_cx prev_cy prev_area prev_ratio"
).split()
assert len(STATE_FIELDS) == QX_STATE_WORDS
# flight_mode != 0: the outer loops' (integral, previous error) memory and the position row of the state snapshot
CASCADE_FIELDS = (
    "att_i0 att_i1 att_i2 att_e0 att_e1 att_e2 vel_i0 vel_i1 vel_e0 vel_e1 pos_i0 pos_i1 pos_e0 pos_e1 zv_i zv_e zp_i zp_e "
    "s_px s_py s_pz pad0 pad1 pad2"
).split()
assert len(STATE_FIELDS) + len(CASCADE_FIELDS) == QX_STATE_WORDS_CASCADE
_INT_FIELDS = {"step_count": np.int32, "rng_ctr": np.uint32, "flags": np.uint32}


def _expect_aligned(t: torch.Tensor, name: str, nbytes: int) -> None:
    """Raise ValueError naming `name` unless `t` starts on an `nbytes` boundary: the kernels access it with vector
    instructions of that width (include/quadx_b200.h, Conventions), which fault on a misaligned address."""
    if t.data_ptr() % nbytes:
        raise ValueError(f"{name}: the kernels access this buffer with {nbytes}-byte vectors, so it must start on a {nbytes}-byte "
                         f"boundary; got address {t.data_ptr():#x} (a column view such as buf[:, 1:21] is offset by its first column)")


class Box:
    """Minimal stand-in for ``gymnasium.spaces.Box`` (hover.py:59-70)."""

    def __init__(self, low, high, dtype=np.float64):
        self.low = np.asarray(low, dtype=dtype)
        self.high = np.asarray(high, dtype=dtype)
        self.shape = self.low.shape
        self.dtype = np.dtype(dtype)

    def sample(self, rng: np.random.Generator | None = None):
        rng = rng or np.random.default_rng()
        lo = np.where(np.isfinite(self.low), self.low, -1.0)
        hi = np.where(np.isfinite(self.high), self.high, 1.0)
        return rng.uniform(lo, hi).astype(self.dtype)

    def contains(self, x) -> bool:
        x = np.asarray(x)
        return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))

    def __repr__(self):
        return f"Box({self.low.min()}, {self.high.max()}, {self.shape}, {self.dtype})"


class QuadXSim:
    """Thin owner of one ``QxHandle``: tensors in, tensors out, current torch stream."""

    def __init__(self, n_envs: int, cfg: QxConfig | None = None, seed: int = 0, env_id0: int = 0,
                 device: int | torch.device | None = None, task: int = QX_TASK_HOVER):
        if not torch.cuda.is_available():
            raise RuntimeError("QuadXSim needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = _lib.lib()
        self.device = _lib.cuda_device(device)
        self.cfg = cfg if cfg is not None else default_config(task)
        self.n = int(n_envs)
        h = C.c_void_p()
        check(self.lib.qx_create(C.byref(self.cfg), self.n, C.c_uint64(seed), C.c_uint64(env_id0), self.device.index, C.byref(h)))
        self._h = h
        self.obs_dim = int(self.lib.qx_obs_dim(h))
        self.act_dim = int(self.lib.qx_act_dim(h))

    # -- lifetime ----------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None):
            self.lib.qx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _obs_layout(self, obs: torch.Tensor | None) -> tuple[int, int]:
        if obs is None:
            return 0, QX_OBS_F32
        if obs.device != self.device or obs.dim() != 2 or obs.shape[0] != self.n or obs.stride(1) != 1 or obs.shape[1] < self.obs_dim:
            raise ValueError("obs: expected [n_envs, >=obs_dim] with unit inner stride on the sim device")
        if obs.dtype not in (torch.float32, torch.bfloat16):
            raise TypeError("obs buffer must be float32 or bfloat16")
        if obs.stride(0) % 4 == 0:  # rows written as 16-byte (f32) / 8-byte (bf16) vectors; other strides element by element
            _expect_aligned(obs, "obs", 4 * obs.element_size())
        return obs.stride(0), QX_OBS_F32 if obs.dtype == torch.float32 else QX_OBS_BF16

    # -- device API ----------------------------------------------------------------
    def reset(self, obs: torch.Tensor | None = None, mask: torch.Tensor | None = None) -> None:
        """qx_reset: obs [n, >=obs_dim] f32/bf16 (row stride = obs.stride(0)), mask u8/bool [n]."""
        stride, code = self._obs_layout(obs)
        if mask is not None:
            if mask.dtype == torch.bool:
                mask = mask.view(torch.uint8)
            expect(mask, "mask", dtype=torch.uint8, device=self.device, shape=(self.n,))
        check(self.lib.qx_reset(self._h, ptr(mask), ptr(obs), code, stride, stream(self.device)))

    def _step_args(self, actions, obs, reward, terminated, truncated, terminal_obs) -> tuple:
        expect(actions, "actions", dtype=torch.float32, device=self.device, shape=(self.n, self.act_dim))
        expect(reward, "reward", dtype=torch.float32, device=self.device, shape=(self.n,))
        expect(terminated, "terminated", dtype=torch.uint8, device=self.device, shape=(self.n,))
        expect(truncated, "truncated", dtype=torch.uint8, device=self.device, shape=(self.n,))
        if self.act_dim == 4:
            _expect_aligned(actions, "actions", 16)  # one float4 per env
        stride, code = self._obs_layout(obs)
        if terminal_obs is not None:
            expect(terminal_obs, "terminal_obs", dtype=torch.float32, device=self.device, shape=(self.n, self.obs_dim))
            _expect_aligned(terminal_obs, "terminal_obs", 16)
        return (self._h, ptr(actions), ptr(obs), code, stride, ptr(reward), ptr(terminated), ptr(truncated), ptr(terminal_obs),
                stream(self.device))

    def step(self, actions: torch.Tensor, obs: torch.Tensor | None, reward: torch.Tensor, terminated: torch.Tensor,
             truncated: torch.Tensor, terminal_obs: torch.Tensor | None = None, split: bool = False) -> None:
        """qx_step on the current stream; all buffers are caller-owned device tensors.  ``split=True`` issues the two
        halves step_begin + step_end (the deferred reset-queue path the PPO rollout uses) instead of qx_step, which
        resets finished envs inside the step launch for small batches."""
        if split:
            self.step_begin(actions, obs, reward, terminated, truncated, terminal_obs)
            self.step_end(obs)
            return
        check(self.lib.qx_step(*self._step_args(actions, obs, reward, terminated, truncated, terminal_obs)))

    def step_begin(self, actions: torch.Tensor, obs: torch.Tensor | None, reward: torch.Tensor, terminated: torch.Tensor,
                   truncated: torch.Tensor, terminal_obs: torch.Tensor | None = None) -> None:
        """qx_step_begin, the first half of step(split=True): the step, with the finished envs queued (done_queue) for step_end."""
        check(self.lib.qx_step_begin(*self._step_args(actions, obs, reward, terminated, truncated, terminal_obs)))

    def step_end(self, obs: torch.Tensor | None) -> None:
        """qx_step_end: re-create the envs step_begin queued and write their first observation."""
        stride, code = self._obs_layout(obs)
        check(self.lib.qx_step_end(self._h, ptr(obs), code, stride, stream(self.device)))

    def done_queue(self) -> tuple[C.c_void_p, C.c_void_p]:
        """qx_done_queue: the fixed device addresses of (count, env indices) of the envs the last step_begin queued."""
        cnt, idx = C.c_void_p(), C.c_void_p()
        check(self.lib.qx_done_queue(self._h, C.byref(cnt), C.byref(idx)))
        return cnt, idx

    def step_k(self, actions: torch.Tensor, obs: torch.Tensor | None, reward: torch.Tensor, terminated: torch.Tensor,
               truncated: torch.Tensor) -> None:
        k = actions.shape[0]
        expect(actions, "actions", dtype=torch.float32, device=self.device, shape=(k, self.n, self.act_dim))
        if self.act_dim == 4:
            _expect_aligned(actions, "actions", 16)
        if obs is not None:
            expect(obs, "obs", dtype=torch.float32, device=self.device, shape=(k, self.n, self.obs_dim))
            _expect_aligned(obs, "obs", 16)
        expect(reward, "reward", dtype=torch.float32, device=self.device, shape=(k, self.n))
        expect(terminated, "terminated", dtype=torch.uint8, device=self.device, shape=(k, self.n))
        expect(truncated, "truncated", dtype=torch.uint8, device=self.device, shape=(k, self.n))
        check(self.lib.qx_step_k(self._h, k, ptr(actions), ptr(obs), ptr(reward), ptr(terminated), ptr(truncated), stream(self.device)))

    def render(self, env_idx: torch.Tensor | Sequence[int] | None = None, fmt: str = "rgba", out: torch.Tensor | None = None) -> torch.Tensor:
        """qx_render: the FPV camera frames of the envs' current poses (those the last observation's camera columns were
        computed from), u8 on the sim device, on the current stream.  fmt "rgba" -> [m, res, res, 4] (the layout of the
        reference's rgbaImg), "mask" -> [m, res, res] (255 on the red box: the mask detect_rectangle starts from).
        env_idx: int32 CUDA tensor or sequence of ints (an index outside [0, n) gives a background frame); None = every env.
        out: optional caller-owned buffer of that shape."""
        code = {"rgba": QX_FRAME_RGBA, "mask": QX_FRAME_MASK}.get(fmt)
        if code is None:
            raise ValueError(f"fmt must be 'rgba' or 'mask', got {fmt!r}")
        if env_idx is not None:
            if isinstance(env_idx, torch.Tensor):
                expect(env_idx, "env_idx", dtype=torch.int32, device=self.device, shape=(env_idx.numel(),))
            else:
                env_idx = torch.tensor(list(env_idx), dtype=torch.int32, device=self.device)
        m = self.n if env_idx is None else env_idx.numel()
        res = int(self.cfg.cam_res)
        shape = (m, res, res, 4) if code == QX_FRAME_RGBA else (m, res, res)
        if out is None:
            out = torch.empty(shape, dtype=torch.uint8, device=self.device)
        else:
            expect(out, "out", dtype=torch.uint8, device=self.device, shape=shape)
        check(self.lib.qx_render(self._h, ptr(env_idx), m, code, ptr(out), stream(self.device)))
        return out

    def episode_record(self, ret: torch.Tensor, length: torch.Tensor, end: torch.Tensor, n_closed: torch.Tensor) -> None:
        """qx_episode_record on the current stream (a sim with auto_reset = 0, after every step): the open records (end == 0)
        of envs whose episode has ended are closed with the episode's return (f32 [n]), length (int32 [n]) and flags word
        (int32 [n], the bits of qx_get_flags, never 0 once closed); n_closed (int32 [1]) counts the closed records.  Zero
        `end` and `n_closed` before the first step of an evaluation."""
        expect(ret, "ret", dtype=torch.float32, device=self.device, shape=(self.n,))
        expect(length, "length", dtype=torch.int32, device=self.device, shape=(self.n,))
        expect(end, "end", dtype=torch.int32, device=self.device, shape=(self.n,))  # u32 words on the device; the flag bits stay below bit 31
        expect(n_closed, "n_closed", dtype=torch.int32, device=self.device, shape=(1,))
        check(self.lib.qx_episode_record(self._h, ptr(ret), ptr(length), ptr(end), ptr(n_closed), stream(self.device)))

    # -- host API ----------------------------------------------------------------
    def reset_host(self, mask: np.ndarray | None = None) -> np.ndarray:
        obs = np.empty((self.n, self.obs_dim), np.float32)
        m = None
        if mask is not None:
            m = np.ascontiguousarray(mask, dtype=np.uint8)
            obs[:] = 0.0
        check(self.lib.qx_reset_host(self._h, None if m is None else m.ctypes.data_as(C.c_void_p), obs.ctypes.data_as(C.c_void_p)))
        return obs

    def step_host(self, actions: np.ndarray, want_terminal_obs: bool = False):
        a = np.ascontiguousarray(actions, dtype=np.float32).reshape(self.n, self.act_dim)
        obs = np.empty((self.n, self.obs_dim), np.float32)
        rew = np.empty(self.n, np.float32)
        te = np.empty(self.n, np.uint8)
        tr = np.empty(self.n, np.uint8)
        tobs = np.zeros((self.n, self.obs_dim), np.float32) if want_terminal_obs else None
        check(self.lib.qx_step_host(self._h, a.ctypes.data_as(C.c_void_p), obs.ctypes.data_as(C.c_void_p),
                                    rew.ctypes.data_as(C.c_void_p), te.ctypes.data_as(C.c_void_p), tr.ctypes.data_as(C.c_void_p),
                                    None if tobs is None else tobs.ctypes.data_as(C.c_void_p)))
        return obs, rew, te.astype(bool), tr.astype(bool), tobs

    def step_host_tensors(self, actions: torch.Tensor, obs: torch.Tensor, reward: torch.Tensor, terminated: torch.Tensor,
                          truncated: torch.Tensor) -> None:
        """qx_step_host_ex on caller-owned CPU tensors (pinned ones are read / written in place by the copy engines):
        `obs` is float32 or bfloat16 [n, obs_dim] -- bfloat16 halves the bytes of the device-to-host copy that bounds this call."""
        for t, shape, dt, name in ((actions, (self.n, self.act_dim), torch.float32, "actions"), (obs, (self.n, self.obs_dim), (torch.float32, torch.bfloat16), "obs"),
                                   (reward, (self.n,), torch.float32, "reward"), (terminated, (self.n,), torch.uint8, "terminated"),
                                   (truncated, (self.n,), torch.uint8, "truncated")):
            expect(t, name, dtype=dt, device=torch.device("cpu"), shape=shape)
        check(self.lib.qx_step_host_ex(self._h, ptr(actions), ptr(obs), 1 if obs.dtype == torch.bfloat16 else 0, ptr(reward), ptr(terminated),
                                       ptr(truncated), None))

    @property
    def state_fields(self) -> list[str]:
        """Names of the carried words, in plane order (qx_state_words of them)."""
        fields = STATE_FIELDS + CASCADE_FIELDS if self.cfg.flight_mode != 0 else STATE_FIELDS
        assert len(fields) == self.lib.qx_state_words(self._h)
        return fields

    def get_state(self) -> dict[str, np.ndarray]:
        torch.cuda.synchronize(self.device)
        fields = self.state_fields
        raw = np.empty((len(fields), self.n), np.float32)
        check(self.lib.qx_get_state(self._h, raw.ctypes.data_as(C.c_void_p)))
        out = {}
        for k, name in enumerate(fields):
            out[name] = raw[k].view(_INT_FIELDS[name]).copy() if name in _INT_FIELDS else raw[k].copy()
        return out

    def set_state(self, state: dict[str, np.ndarray]) -> None:
        torch.cuda.synchronize(self.device)
        fields = self.state_fields
        raw = np.zeros((len(fields), self.n), np.float32)
        for k, name in enumerate(fields):
            v = np.asarray(state[name])
            raw[k] = v.astype(_INT_FIELDS[name]).view(np.float32) if name in _INT_FIELDS else v.astype(np.float32)
        check(self.lib.qx_set_state(self._h, raw.ctypes.data_as(C.c_void_p)))

    def flags(self, first: int = 0, count: int | None = None) -> np.ndarray:
        """The flags word of envs [first, first + count) (qx_get_flags): one word per env, no full-state transfer."""
        torch.cuda.synchronize(self.device)
        count = self.n - first if count is None else count
        out = np.empty(count, np.uint32)
        check(self.lib.qx_get_flags(self._h, first, count, out.ctypes.data_as(C.c_void_p)))
        return out

    def nonfinite_count(self) -> int:
        """Envs terminated because their state stopped being finite (failure containment)."""
        torch.cuda.synchronize(self.device)
        n = C.c_int64()
        check(self.lib.qx_nonfinite_count(self._h, C.byref(n)))
        return n.value

    def episode_stats(self, clear: bool = True) -> tuple[float, int, int]:
        torch.cuda.synchronize(self.device)
        s, l, n = C.c_double(), C.c_int64(), C.c_int64()
        check(self.lib.qx_episode_stats(self._h, C.byref(s), C.byref(l), C.byref(n), int(clear)))
        return s.value, l.value, n.value


class QuadXHoverVecEnv:
    """SB3-``VecEnv``-shaped batched hover env (train_hover.py:42).

    ``reset()`` / ``step(actions)`` take and return torch tensors on the GPU:
    obs f32 [N,20], rewards f32 [N], dones bool [N].  ``infos`` is built lazily:
    it is a list of per-env dicts only for the envs that finished (SB3 only
    reads ``terminal_observation``, ``TimeLimit.truncated`` and ``episode``
    there); pass ``infos=False`` to skip the host round trip entirely.
    """

    def __init__(self, num_envs: int, seed: int = 0, device=None, cfg: QxConfig | None = None, env_id0: int = 0,
                 infos: bool = True, **cfg_overrides: Any):
        cfg = cfg if cfg is not None else default_config(QX_TASK_HOVER)
        cfg.update(auto_reset=1, **cfg_overrides)
        self.sim = QuadXSim(num_envs, cfg, seed=seed, env_id0=env_id0, device=device)
        self.num_envs = num_envs
        self.device = self.sim.device
        self.observation_space = Box(-np.inf * np.ones(20), np.inf * np.ones(20), np.float64)  # hover.py:67-70
        self.action_space = Box(-np.ones(4), np.ones(4), np.float64)  # hover.py:59-61
        n, d = num_envs, self.device
        self.obs = torch.zeros(n, 20, device=d)
        self.rewards = torch.zeros(n, device=d)
        self.terminated = torch.zeros(n, dtype=torch.uint8, device=d)
        self.truncated = torch.zeros(n, dtype=torch.uint8, device=d)
        self.terminal_obs = torch.zeros(n, 20, device=d)
        self._actions = None
        self._want_infos = infos
        self._ep_ret = torch.zeros(n, device=d)
        self._ep_len = torch.zeros(n, dtype=torch.int32, device=d)
        self.render_mode = None

    # -- VecEnv API ----------------------------------------------------------------
    def reset(self) -> torch.Tensor:
        self.sim.reset(self.obs)
        self._ep_ret.zero_()
        self._ep_len.zero_()
        return self.obs

    def step_async(self, actions) -> None:
        a = torch.as_tensor(actions, dtype=torch.float32, device=self.device).reshape(self.num_envs, 4)
        self._actions = a.contiguous()

    def step_wait(self):
        self.sim.step(self._actions, self.obs, self.rewards, self.terminated, self.truncated, self.terminal_obs)
        dones = (self.terminated | self.truncated).bool()
        infos: list[dict] | None = None
        if self._want_infos:
            self._ep_ret += self.rewards
            self._ep_len += 1
            infos = [{} for _ in range(self.num_envs)]
            idx = torch.nonzero(dones).flatten()
            if idx.numel():
                tobs = self.terminal_obs[idx].cpu().numpy()
                trunc_only = (self.truncated[idx].bool() & ~self.terminated[idx].bool()).cpu().numpy()
                r, l = self._ep_ret[idx].cpu().numpy(), self._ep_len[idx].cpu().numpy()
                for j, i in enumerate(idx.cpu().numpy()):
                    infos[i] = {
                        "terminal_observation": tobs[j],
                        "TimeLimit.truncated": bool(trunc_only[j]),
                        "episode": {"r": float(r[j]), "l": int(l[j])},
                    }
                self._ep_ret[idx] = 0.0
                self._ep_len[idx] = 0
        return self.obs, self.rewards, dones, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def close(self) -> None:
        self.sim.close()

    def seed(self, seed=None):
        return [None] * self.num_envs

    def get_attr(self, name, indices=None):
        return [getattr(self, name)] * self.num_envs

    def set_attr(self, name, value, indices=None):
        setattr(self, name, value)

    def env_method(self, method_name, *args, indices=None, **kwargs):
        raise NotImplementedError("the batched env has no per-env Python objects")

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [False] * self.num_envs

    def episode_stats(self, clear: bool = True):
        """(sum of returns, sum of lengths, count) of the episodes finished since the last call."""
        return self.sim.episode_stats(clear)


class QuadXHoverEnv:
    """Single-env facade with the reference's gymnasium signatures (hover.py:10-365).

    ``flight_mode`` and ``agent_hz`` are accepted like the reference's
    constructor (hover.py:11-16); the reference ignores ``flight_mode``
    (``set_mode(0)`` is literal, hover.py:92) and so does this class, unless
    ``honour_flight_mode=True`` is passed: then the drone flies in that PyFlyt
    mode (-1..7, the outer PID loops of cf2x.yaml:21-54; set ``action_scale`` /
    ``thrust_scale`` / ``thrust_bias`` to map the Box(-1, 1) action onto it).

    ``render_mode="rgb_array"`` makes ``render()`` return the FPV camera frame of the current state (``np.uint8``
    [res, res, 4], what the reference's ``drones[0].rgbaImg`` holds).  It is unrelated to ``render``, which is hover.py's
    switch of the floor rule (hover.py:283).
    """

    metadata = {"render_modes": ["rgb_array"]}

    def __init__(self, flight_mode: int = 0, agent_hz: int = 40, render: bool = False, seed: int = 0, device=None,
                 honour_flight_mode: bool = False, render_mode: str | None = None, **cfg_overrides):
        if render_mode not in (None, "rgb_array"):
            raise ValueError(f"render_mode must be None or 'rgb_array', got {render_mode!r}")
        self.render_mode = render_mode
        self.flight_mode = flight_mode
        self.agent_hz = agent_hz
        cfg = default_config(QX_TASK_HOVER)
        if honour_flight_mode:
            cfg_overrides.setdefault("flight_mode", int(flight_mode))
        cfg.update(auto_reset=0, render=int(render), agent_dt=1.0 / agent_hz,
                   aviary_steps_per_step=int(cfg.physics_hz / agent_hz), **cfg_overrides)
        self.sim = QuadXSim(1, cfg, seed=seed, device=device)
        self.action_space = Box(-np.ones(4), np.ones(4), np.float64)  # hover.py:59-61
        self.observation_space = Box(-np.inf * np.ones(20), np.inf * np.ones(20), np.float64)  # hover.py:67-70
        self.info = {"out_of_bounds": False, "collision": False, "env_complete": False, "on_floor": False}  # hover.py:53-57
        self.state = np.zeros(20)

    def reset(self, seed=None, options=None):
        obs = self.sim.reset_host()
        self.info = {"out_of_bounds": False, "collision": False, "env_complete": False, "on_floor": False}  # hover.py:102
        self.state = obs[0].astype(np.float64)
        return self.state, self.info

    def step(self, action):
        a = np.asarray(action, dtype=np.float32).reshape(1, 4)
        obs, rew, te, tr, _ = self.sim.step_host(a)
        flags = int(self.sim.flags()[0])
        self.info["out_of_bounds"] = bool(flags & 8)  # hover.py:280
        self.info["on_floor"] = bool(flags & 16)  # hover.py:289
        self.state = obs[0].astype(np.float64)
        return self.state, float(rew[0]), bool(te[0]), bool(tr[0]), self.info

    def render(self):
        if self.render_mode != "rgb_array":
            raise NotImplementedError("rendering is out of scope (SURVEY 2, row 6/11)")
        return self.sim.render().cpu().numpy()[0]

    def close(self):
        self.sim.close()
