"""On-device PPO for the batched hover env: what ``train_hover.py:40-63`` does with
stable-baselines3 (vec env -> VecNormalize -> MlpPolicy [128,128] -> learn ->
checkpoints), with the rollout half (policy forward, sampling, reward /
observation normalisation, GAE) on the hand-written kernels of
``include/ppo_b200.h`` and no host round trip per env step.

The update half (SB3 ``PPO.train``) runs on the hand-written kernels too
(``FusedUpdater``: forward + loss + backward of both networks in one tcgen05
kernel, gradient reduction, clip + Adam + bf16 re-pack; csrc/ppo_update_kernels.cu);
its only collective is one all-reduce of the flat 39 049-float gradient per
optimiser step (``torch.distributed``, NCCL), captured into the same CUDA graph
as the kernels.  A plain-PyTorch autograd update is kept as the reference the
tests compare against (``PPOConfig.fused_update=False``).

Hyper-parameter names and defaults follow SB3 PPO / VecNormalize (SURVEY 9.5).
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass

import torch
import torch.distributed as dist
from torch import nn

from . import _lib
from ._lib import PpoPolicy, QxConfig, check, default_config, expect, ptr, stream
from .hover_env import QuadXSim

HID, IN_PAD, HEAD_PAD = 128, 32, 16


def _capture(body, device) -> torch.cuda.CUDAGraph:
    """Capture `body` into a CUDA graph on a fresh side stream forked from, and joined back into, the current stream."""
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream(device))
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        body()
    torch.cuda.current_stream(device).wait_stream(side)
    return g


class ActorCritic(nn.Module):
    """SB3 ``MlpPolicy`` with ``net_arch=[128, 128]`` (train_hover.py:57): separate
    tanh MLPs for the actor and the critic, state-independent ``log_std``,
    orthogonal init (gain sqrt 2; 0.01 on the action head; 1 on the value head).

    ``hidden`` < 128 (SB3's default ``net_arch=[64, 64]``, what the yaw config of SURVEY 8d C3 would train) is held as an
    exact embedding in the 128-wide layers the kernels are tiled for: the extra rows / columns and biases are zero, so the
    extra units output tanh(0) = 0, receive a zero back-propagated signal (their outgoing weights are zero) and a zero weight
    gradient (their activations are zero) -- Adam never moves them and the global gradient norm does not see them.  Forward,
    gradients and the trajectory of training are those of the narrow network (``tests/test_gpu_update.py``)."""

    def __init__(self, obs_dim: int = 20, act_dim: int = 4, log_std_init: float = 0.0, hidden: int = HID):
        super().__init__()
        assert obs_dim <= IN_PAD and act_dim <= 4 and 0 < hidden <= HID
        self.obs_dim, self.act_dim, self.hidden = obs_dim, act_dim, hidden
        self.pi1, self.pi2, self.mu = nn.Linear(obs_dim, HID), nn.Linear(HID, HID), nn.Linear(HID, act_dim)
        self.vf1, self.vf2, self.v = nn.Linear(obs_dim, HID), nn.Linear(HID, HID), nn.Linear(HID, 1)
        self.log_std = nn.Parameter(torch.full((act_dim,), float(log_std_init)))
        h = hidden
        for lin, gain, rows, cols in ((self.pi1, math.sqrt(2), h, obs_dim), (self.pi2, math.sqrt(2), h, h), (self.vf1, math.sqrt(2), h, obs_dim),
                                      (self.vf2, math.sqrt(2), h, h), (self.mu, 0.01, act_dim, h), (self.v, 1.0, 1, h)):
            w = torch.empty(rows, cols)
            nn.init.orthogonal_(w, gain=gain)
            with torch.no_grad():
                lin.weight.zero_()
                lin.weight[:rows, :cols].copy_(w)
            nn.init.zeros_(lin.bias)

    def num_effective_params(self) -> int:
        h, od, ad = self.hidden, self.obs_dim, self.act_dim
        return 2 * (od * h + h + h * h + h) + (h * ad + ad) + (h + 1) + ad

    def forward(self, obs: torch.Tensor):
        hp = torch.tanh(self.pi2(torch.tanh(self.pi1(obs))))
        hv = torch.tanh(self.vf2(torch.tanh(self.vf1(obs))))
        return self.mu(hp), self.v(hv).squeeze(-1)

    def evaluate_actions(self, obs: torch.Tensor, actions: torch.Tensor):
        mean, value = self(obs)
        std = self.log_std.exp()
        z = (actions - mean) / std
        logp = (-0.5 * z * z - self.log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
        entropy = (0.5 + 0.5 * math.log(2 * math.pi) + self.log_std).sum().expand_as(logp)
        return value, logp, entropy


# stable-baselines3 ActorCriticPolicy parameter names (net_arch=[128,128], separate pi / vf MLPs) -> ActorCritic modules
SB3_KEYS = {
    "mlp_extractor.policy_net.0": "pi1", "mlp_extractor.policy_net.2": "pi2", "action_net": "mu",
    "mlp_extractor.value_net.0": "vf1", "mlp_extractor.value_net.2": "vf2", "value_net": "v",
}


def export_sb3_state_dict(model: "ActorCritic") -> dict:
    """Policy weights under stable-baselines3's parameter names, so that `policy.load_state_dict(...)` of an SB3
    `ActorCriticPolicy(net_arch=[128, 128])` (what train_hover.py:47-58 builds with PPO) accepts them -- the
    counterpart of `model.save` in train_hover.py:26,62 for users who play the policy back with SB3
    (test_hover.py:8-21)."""
    sd = {"log_std": model.log_std.detach().cpu().clone()}
    h = getattr(model, "hidden", HID)
    for sb3, mine in SB3_KEYS.items():
        lin = getattr(model, mine)
        w, b = lin.weight.detach().cpu(), lin.bias.detach().cpu()
        rows = h if w.shape[0] == HID else w.shape[0]  # a narrow net_arch lives in the top-left block of the 128-wide layers
        cols = h if w.shape[1] == HID else w.shape[1]
        sd[f"{sb3}.weight"] = w[:rows, :cols].clone()
        sd[f"{sb3}.bias"] = b[:rows].clone()
    return sd


def import_sb3_state_dict(model: "ActorCritic", sd: dict) -> None:
    with torch.no_grad():
        model.log_std.copy_(sd["log_std"])
        for sb3, mine in SB3_KEYS.items():
            lin, w, b = getattr(model, mine), sd[f"{sb3}.weight"], sd[f"{sb3}.bias"]
            lin.weight.zero_(); lin.bias.zero_()
            lin.weight[:w.shape[0], :w.shape[1]].copy_(w)
            lin.bias[:b.shape[0]].copy_(b)


def export_vecnormalize(obs_stats: "RunningStats", ret_stats: "RunningStats", cfg: "PPOConfig") -> dict:
    """The fields of SB3's VecNormalize pickle (`env.save`, train_hover.py:27,63): obs_rms / ret_rms
    {mean, var, count}, clip_obs, clip_reward, gamma, epsilon, norm_obs, norm_reward."""
    def rms(st):
        s, d = st.stats.detach().cpu().numpy(), st.dim
        return {"mean": s[:d].copy(), "var": s[d:2 * d].copy(), "count": float(s[2 * d])}
    return {"obs_rms": rms(obs_stats), "ret_rms": rms(ret_stats), "clip_obs": cfg.clip_obs, "clip_reward": cfg.clip_reward,
            "gamma": cfg.gamma, "epsilon": obs_stats.eps, "norm_obs": cfg.norm_obs, "norm_reward": cfg.norm_reward}


def export_sb3_zip(model: "ActorCritic", path: str, vecnormalize: dict | None = None, sb3_version: str = "2.7.0", hyper: dict | None = None) -> None:
    """Write the policy the way stable-baselines3's `save_to_zip_file` lays out a model archive: `policy.pth` (the
    `ActorCriticPolicy` state dict under SB3's parameter names), `_stable_baselines3_version` (the version the reference
    pins, uv.lock:990), `system_info.txt`, and a `data` entry.  SB3's own `data` holds cloudpickles of gymnasium / SB3
    objects (spaces, schedules, the policy class); neither package exists where this runs, so `data` here is plain JSON
    with the constructor arguments (net_arch, log_std_init, PPO hyper-parameters, spaces as shape / bounds, timesteps).
    `vecnormalize` (export_vecnormalize) goes in as `vecnormalize.npz`.

    tools/load_into_sb3.py, run on the reference side, rebuilds `PPO("MlpPolicy", VecNormalize(DummyVecEnv(QuadXHoverEnv)))`
    from these entries with public SB3 API and writes the `.zip` + `.pkl` pair the reference's playback loads
    (test_hover.py:8-11)."""
    import io
    import json
    import zipfile

    import numpy as np

    hyper = dict(hyper or {})
    data = {"policy_class": "stable_baselines3.common.policies.ActorCriticPolicy", "algorithm": "PPO",
            "policy_kwargs": {"net_arch": [getattr(model, "hidden", HID)] * 2, "log_std_init": float(hyper.pop("log_std_init", 0.0)), "activation_fn": "torch.nn.Tanh"},
            "observation_space": {"type": "Box", "shape": [model.obs_dim], "low": "-inf", "high": "inf", "dtype": "float64"},  # hover.py:67-70
            "action_space": {"type": "Box", "shape": [model.act_dim], "low": -1.0, "high": 1.0, "dtype": "float64"},           # hover.py:59-61
            "learning_rate": 3e-4, "n_steps": 2048, "batch_size": 64, "gamma": 0.99, "gae_lambda": 0.95, "clip_range": 0.2, "ent_coef": 0.0,
            "vf_coef": 0.5, "max_grad_norm": 0.5, "num_timesteps": 0}
    data.update(hyper)
    with zipfile.ZipFile(path, "w") as z:
        buf = io.BytesIO()
        torch.save(export_sb3_state_dict(model), buf)
        z.writestr("policy.pth", buf.getvalue())
        z.writestr("data", json.dumps(data, indent=1))
        z.writestr("_stable_baselines3_version", sb3_version)
        z.writestr("system_info.txt", "exported by fpv_drone_rl_agent_b200 (B200 on-device PPO); see tools/load_into_sb3.py\n")
        if vecnormalize is not None:
            buf = io.BytesIO()
            flat = {}
            for k, v in vecnormalize.items():
                if isinstance(v, dict):
                    for kk, vv in v.items():
                        flat[f"{k}.{kk}"] = np.asarray(vv)
                else:
                    flat[k] = np.asarray(v)
            np.savez(buf, **flat)
            z.writestr("vecnormalize.npz", buf.getvalue())


class PackedPolicy:
    """bf16 copy of an ``ActorCritic`` in the layout of ``struct PpoPolicy``."""

    def __init__(self, model: ActorCritic, device):
        self.model, self.device = model, _lib.cuda_device(device)
        d = self.device
        self.w1 = torch.zeros(2 * HID, IN_PAD, dtype=torch.bfloat16, device=d)
        self.w2p = torch.zeros(HID, HID, dtype=torch.bfloat16, device=d)
        self.w2v = torch.zeros(HID, HID, dtype=torch.bfloat16, device=d)
        self.w3 = torch.zeros(HEAD_PAD, 2 * HID, dtype=torch.bfloat16, device=d)
        self.b1 = torch.zeros(2 * HID, device=d)
        self.b2 = torch.zeros(2 * HID, device=d)
        self.b3 = torch.zeros(HEAD_PAD, device=d)
        self.log_std = torch.zeros(4, device=d)
        self.struct = PpoPolicy(self.w1.data_ptr(), self.w2p.data_ptr(), self.w2v.data_ptr(), self.w3.data_ptr(), self.b1.data_ptr(),
                                self.b2.data_ptr(), self.b3.data_ptr(), self.log_std.data_ptr(), model.obs_dim, model.act_dim)
        self.refresh()

    @torch.no_grad()
    def refresh(self) -> None:
        """Re-pack after an optimiser step (a handful of tiny copies, stream-ordered)."""
        m, od, ad = self.model, self.model.obs_dim, self.model.act_dim
        self.w1[:HID, :od].copy_(m.pi1.weight)
        self.w1[HID:, :od].copy_(m.vf1.weight)
        self.w2p.copy_(m.pi2.weight)
        self.w2v.copy_(m.vf2.weight)
        self.w3[:ad, :HID].copy_(m.mu.weight)
        self.w3[ad, HID:].copy_(m.v.weight[0])
        self.b1[:HID].copy_(m.pi1.bias)
        self.b1[HID:].copy_(m.vf1.bias)
        self.b2[:HID].copy_(m.pi2.bias)
        self.b2[HID:].copy_(m.vf2.bias)
        self.b3[:ad].copy_(m.mu.bias)
        self.b3[ad].copy_(m.v.bias[0])
        self.log_std[:ad].copy_(m.log_std)


class RunningStats:
    """VecNormalize ``RunningMeanStd`` kept on the device: {mean[dim], var[dim], count} in fp64."""

    def __init__(self, dim: int, device, eps: float = 1e-8):
        self.stats = torch.zeros(2 * dim + 1, dtype=torch.float64, device=device)
        self.dim, self.eps, self.device = dim, eps, self.stats.device  # device with its index; CPU statistics serve export / gloo tests
        self.stats[dim:2 * dim] = 1.0
        self.stats[2 * dim] = 1e-4  # RunningMeanStd(epsilon=1e-4)
        self.mean = torch.zeros(dim, device=device)
        self.inv_std = torch.ones(dim, device=device)
        self.scratch = torch.zeros(_lib.lib().ppo_running_stats_scratch_bytes(dim) // 8, dtype=torch.float64, device=device)

    def update(self, x: torch.Tensor, out: tuple | None = None) -> None:
        """Merge the rows of x; the refreshed fp32 (mean, inv_std) go to `out` instead of self.mean / self.inv_std when given."""
        assert x.dtype == torch.float32 and x.dim() == 2 and x.shape[1] >= self.dim and x.stride(1) == 1
        mean, inv_std = out if out is not None else (self.mean, self.inv_std)
        check(_lib.lib().ppo_running_stats_update(ptr(x), x.stride(0), x.shape[0], self.dim, ptr(self.stats), self.eps, ptr(mean),
                                                  ptr(inv_std), ptr(self.scratch), stream(self.device)))

    def state_dict(self):
        return {"stats": self.stats.clone(), "mean": self.mean.clone(), "inv_std": self.inv_std.clone()}

    def load_state_dict(self, sd):
        self.stats.copy_(sd["stats"]); self.mean.copy_(sd["mean"]); self.inv_std.copy_(sd["inv_std"])

    def allreduce_(self) -> None:
        """Merge the replicas' statistics (each saw different envs) -- optional, tiny."""
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return
        d = self.dim
        mean, var, cnt = self.stats[:d].clone(), self.stats[d:2 * d].clone(), self.stats[2 * d].clone()
        tot = cnt.clone()
        dist.all_reduce(tot)
        gmean = mean * cnt
        dist.all_reduce(gmean)
        gmean /= tot
        m2 = (var + (mean - gmean) ** 2) * cnt
        dist.all_reduce(m2)
        self.stats[:d], self.stats[d:2 * d], self.stats[2 * d] = gmean, m2 / tot, tot / dist.get_world_size()  # count per rank: every rank adds its own shard again next rollout
        self.mean.copy_(gmean.float())
        self.inv_std.copy_((1.0 / torch.sqrt(m2 / tot + self.eps)).float())


def policy_forward(pol: PackedPolicy, obs: torch.Tensor, *, obs_stats: RunningStats | None = None, obs_clip: float = 10.0, seed: int = 0,
                   row0: int = 0, step: int = 0, step_base: torch.Tensor | None = None, deterministic: bool = False,
                   actions=None, env_actions=None, values=None, log_probs=None, obs_norm=None, norm: tuple | None = None,
                   update_stats: bool = False, fused_stats: bool = False) -> None:
    """``ActorCriticPolicy.forward`` on the tensor cores (ppo_policy_forward).  norm = (mean, inv_std) overrides obs_stats' buffers.
    update_stats: `obs` is first merged into obs_stats and (mean, inv_std) refreshed -- VecNormalize's ``obs_rms.update`` +
    ``normalize_obs`` of one env step in one call (ppo_policy_forward_stats): two launches chained as programmatic dependents, or,
    with fused_stats, one launch with the merge inside the policy kernel."""
    n = obs.shape[0]
    assert obs.dtype == torch.float32 and obs.stride(1) == 1
    od, ad, dev = pol.model.obs_dim, pol.model.act_dim, pol.device
    for name, t, numel in (("actions", actions, n * ad), ("env_actions", env_actions, n * ad), ("values", values, n),
                           ("log_probs", log_probs, n), ("obs_norm", obs_norm, n * od)):
        if t is not None:
            expect(t, name, dtype=torch.float32, device=dev, numel=numel)
    mean, inv_std = norm if norm is not None else ((obs_stats.mean, obs_stats.inv_std) if obs_stats else (None, None))
    if update_stats:
        assert obs_stats is not None and mean is not None
        check(_lib.lib().ppo_policy_forward_stats(C.byref(pol.struct), ptr(obs), obs.stride(0), n, ptr(obs_stats.stats), obs_stats.eps,
                                                  ptr(obs_stats.scratch), ptr(mean), ptr(inv_std), obs_clip, seed, row0, step, ptr(step_base),
                                                  int(deterministic), ptr(actions), ptr(env_actions), ptr(values), ptr(log_probs), ptr(obs_norm),
                                                  int(fused_stats), stream(pol.device)))
        return
    check(_lib.lib().ppo_policy_forward(C.byref(pol.struct), ptr(obs), obs.stride(0), n, ptr(mean),
                                        ptr(inv_std), obs_clip, seed, row0, step, ptr(step_base),
                                        int(deterministic), ptr(actions), ptr(env_actions), ptr(values), ptr(log_probs), ptr(obs_norm),
                                        stream(pol.device)))


F_TERMINATED, F_TRUNCATED, F_OUT_OF_BOUNDS, F_ON_FLOOR = 2, 4, 8, 16  # bits of the flags word (qx_get_flags)


class PolicyEvaluator:
    """SB3 ``evaluate_policy(model, env, n_eval_episodes, deterministic=True)`` -- the playback loop of test_hover.py:13-27 --
    on the device.  The evaluator owns a sim of ``n_episodes`` envs (auto_reset = 0, env ids 0 .. n_episodes - 1, the caller's
    env config otherwise) and every env flies exactly one episode, so short episodes are not over-represented as they are when
    finished episodes are counted until n_eval_episodes is reached.  Each step is the deterministic policy (a = mean, clipped to
    the action box) on observations normalised with a frozen copy of ``obs_stats`` (VecNormalize with training=False; rewards
    are the raw env rewards, norm_reward=False), the env step, and qx_episode_record, which latches each episode's return,
    length and end flags on the step it ends.

    A chunk of ``chunk`` such steps is one CUDA-graph replay (``use_cuda_graph=False``: eager launches, same results); the host
    reads the number of closed records once per chunk.  Every ``evaluate()`` starts from the state the first reset produced,
    motor-noise counters included, so two evaluations of the same policy give the same numbers.  The packed policy is read
    where it lives: an evaluator built once follows the weights of a policy that keeps training."""

    def __init__(self, policy: PackedPolicy, obs_stats: RunningStats | None, env_cfg=None, n_episodes: int = 4096, seed: int = 0,
                 task: int = 0, obs_clip: float = 10.0, device=None, chunk: int = 32, use_cuda_graph: bool = True):
        if n_episodes <= 0 or chunk <= 0:
            raise ValueError("n_episodes and chunk must be positive")
        cfg = default_config(task) if env_cfg is None else QxConfig.from_buffer_copy(env_cfg)
        if cfg.task != task:
            raise ValueError(f"env_cfg is for task {cfg.task}, the evaluator was asked for task {task}")
        cfg.update(auto_reset=0)
        self.sim = QuadXSim(n_episodes, cfg, seed=seed, env_id0=0, device=policy.device if device is None else device)
        if (policy.struct.obs_dim, policy.struct.act_dim) != (self.sim.obs_dim, self.sim.act_dim):
            self.sim.close()
            raise ValueError(f"policy has obs_dim {policy.struct.obs_dim}, act_dim {policy.struct.act_dim}; task {task} needs "
                             f"{self.sim.obs_dim}, {self.sim.act_dim}")
        if obs_stats is not None and obs_stats.dim != self.sim.obs_dim:
            self.sim.close()
            raise ValueError(f"obs_stats has dim {obs_stats.dim}, task {task} observations have {self.sim.obs_dim}")
        self.pol, self.obs_stats, self.obs_clip = policy, obs_stats, float(obs_clip)
        self.n, self.seed, self.chunk, self.use_cuda_graph = int(n_episodes), int(seed), int(chunk), bool(use_cuda_graph)
        n, d = self.n, self.sim.device
        self.device = d
        self.obs = torch.zeros(n, self.sim.obs_dim, device=d)
        self.env_actions = torch.zeros(n, self.sim.act_dim, device=d)
        self.reward = torch.zeros(n, device=d)
        self.te = torch.zeros(n, dtype=torch.uint8, device=d)
        self.tr = torch.zeros(n, dtype=torch.uint8, device=d)
        self.ret = torch.zeros(n, device=d)
        self.length = torch.zeros(n, dtype=torch.int32, device=d)
        self.end = torch.zeros(n, dtype=torch.int32, device=d)
        self.n_closed = torch.zeros(1, dtype=torch.int32, device=d)
        self.norm = (torch.zeros(self.sim.obs_dim, device=d), torch.ones(self.sim.obs_dim, device=d)) if obs_stats is not None else None
        self.sim.reset(self.obs)
        self._obs0 = self.obs.clone()
        self._state0 = self.sim.get_state()
        self._graph = None
        # one-time kernel attribute setup must not happen inside a graph capture
        policy_forward(self.pol, self.obs, norm=self.norm, obs_clip=self.obs_clip, deterministic=True, env_actions=self.env_actions)

    def _chunk(self) -> None:
        for _ in range(self.chunk):
            policy_forward(self.pol, self.obs, norm=self.norm, obs_clip=self.obs_clip, deterministic=True, env_actions=self.env_actions)
            self.sim.step(self.env_actions, self.obs, self.reward, self.te, self.tr)
            self.sim.episode_record(self.ret, self.length, self.end, self.n_closed)

    def _run_chunk(self) -> None:
        if not self.use_cuda_graph:
            self._chunk()
            return
        if self._graph is None:
            self._graph = _capture(self._chunk, self.device)
        self._graph.replay()

    def evaluate(self) -> tuple[dict, dict]:
        """Fly every env's episode from the initial state.  Returns (summary, records): summary holds evaluate_policy's
        mean_reward / std_reward (population std, as np.std), mean_ep_length, success_rate (truncated by the time limit and not
        terminated), floor_rate (floor rule), oob_rate (left the flight dome), n_episodes and the steps run; records holds
        the per-episode tensors return (f32), length (int32) and end (int32 flags word), one entry per env."""
        self.sim.set_state(self._state0)
        self.obs.copy_(self._obs0)
        if self.norm is not None:
            self.norm[0].copy_(self.obs_stats.mean)
            self.norm[1].copy_(self.obs_stats.inv_std)
        for t in (self.ret, self.length, self.end, self.n_closed):
            t.zero_()
        limit, steps = int(self.sim.cfg.max_steps) + 2, 0  # the hover time limit ends an episode on step max_steps + 2
        while True:
            self._run_chunk()
            steps += self.chunk
            closed = int(self.n_closed.item())
            if closed == self.n:
                break
            if steps >= limit:
                raise RuntimeError(f"{self.n - closed} of {self.n} episodes still open after {steps} steps (every episode ends by step {limit})")
        ret = self.ret.double().cpu()
        end = self.end.cpu()
        trunc, term = (end & F_TRUNCATED) != 0, (end & F_TERMINATED) != 0
        summary = {"mean_reward": float(ret.mean()), "std_reward": float(ret.std(correction=0)),
                   "mean_ep_length": float(self.length.double().mean()), "success_rate": float((trunc & ~term).double().mean()),
                   "floor_rate": float(((end & F_ON_FLOOR) != 0).double().mean()), "oob_rate": float(((end & F_OUT_OF_BOUNDS) != 0).double().mean()),
                   "n_episodes": self.n, "steps": steps}
        return summary, {"return": self.ret.clone(), "length": self.length.clone(), "end": self.end.clone()}

    def close(self) -> None:
        self._graph = None
        self.sim.close()


def evaluate_policy(policy: PackedPolicy, obs_stats: RunningStats | None, env_cfg=None, n_episodes: int = 4096, seed: int = 0,
                    task: int = 0, obs_clip: float = 10.0, device=None, **kw) -> tuple[dict, dict]:
    """One evaluation with a PolicyEvaluator built for it (kw: chunk, use_cuda_graph); (summary, records) as evaluate()."""
    ev = PolicyEvaluator(policy, obs_stats, env_cfg, n_episodes, seed, task, obs_clip, device, **kw)
    try:
        return ev.evaluate()
    finally:
        ev.close()


def gae(rewards, values, dones, last_values, gamma: float, lam: float, advantages, returns) -> None:
    """``RolloutBuffer.compute_returns_and_advantage`` (ppo_gae); all [T, n] contiguous."""
    T, n = rewards.shape
    check(_lib.lib().ppo_gae(ptr(rewards), ptr(values), ptr(dones), ptr(last_values), T, n, gamma, lam, ptr(advantages), ptr(returns),
                             stream(rewards.device)))


def bootstrap_truncated(pol: PackedPolicy, terminal_obs, norm: tuple | None, obs_clip: float, queue: tuple, terminated, truncated,
                        gamma: float, rewards, *, first: bool = False) -> None:
    """SB3's time-limit bootstrap (ppo_bootstrap_truncated): rewards[i] += gamma * V(terminal_obs[i]) for the truncated, not terminated
    envs of the done queue (QuadXSim.done_queue()).  first: rewards[i] = gamma * V(...) instead, for reward_normalize(add=True)."""
    n, dev = terminal_obs.shape[0], pol.device
    expect(terminal_obs, "terminal_obs", dtype=torch.float32, device=dev, shape=(n, pol.model.obs_dim))
    expect(terminated, "terminated", dtype=torch.uint8, device=dev, numel=n)
    expect(truncated, "truncated", dtype=torch.uint8, device=dev, numel=n)
    expect(rewards, "rewards", dtype=torch.float32, device=dev, numel=n)
    mean, inv_std = norm if norm is not None else (None, None)
    fn = _lib.lib().ppo_bootstrap_truncated_first if first else _lib.lib().ppo_bootstrap_truncated
    check(fn(C.byref(pol.struct), ptr(terminal_obs), terminal_obs.stride(0), n, ptr(mean), ptr(inv_std), obs_clip, queue[0], queue[1],
             ptr(terminated), ptr(truncated), gamma, ptr(rewards), stream(dev)))


def reward_normalize(raw_reward, terminated, truncated, returns_acc, ret_stats: RunningStats, gamma: float, clip: float, rewards, dones,
                     *, add: bool = False) -> None:
    """VecNormalize's reward path (ppo_reward_normalize): returns_acc = gamma * returns_acc + raw_reward into ret_stats, rewards =
    clip(raw_reward / std), dones = terminated | truncated.  add: plus what bootstrap_truncated(first=True) stored in rewards."""
    n, dev = raw_reward.shape[0], ret_stats.device
    for name, t, dtype in (("raw_reward", raw_reward, torch.float32), ("terminated", terminated, torch.uint8), ("truncated", truncated, torch.uint8),
                           ("returns_acc", returns_acc, torch.float32), ("rewards", rewards, torch.float32), ("dones", dones, torch.uint8)):
        expect(t, name, dtype=dtype, device=dev, numel=n)
    expect(ret_stats.stats, "ret_stats", dtype=torch.float64, device=dev, numel=3)
    fn = _lib.lib().ppo_reward_normalize_add if add else _lib.lib().ppo_reward_normalize
    check(fn(ptr(raw_reward), ptr(terminated), ptr(truncated), ptr(returns_acc), n, gamma, clip, ret_stats.eps, ptr(ret_stats.stats),
             ptr(rewards), ptr(dones), ptr(ret_stats.scratch), stream(dev)))


def allreduce_gradients(params, world: int) -> None:
    """The one collective of the PPO update: average the flattened gradient (39 049 floats = 156 KB for the
    [128,128] hover policy) over the ranks.  Each rank holds a replica of the policy and a disjoint env shard."""
    if world == 1:
        return
    params = [p for p in params if p.grad is not None]
    flat = torch.cat([p.grad.reshape(-1) for p in params])
    dist.all_reduce(flat)
    flat /= world
    o = 0
    for p in params:
        k = p.numel()
        p.grad.copy_(flat[o:o + k].view_as(p.grad))
        o += k


def shard_env_ids(rank: int, envs_per_rank: int) -> int:
    """First global env id of a rank's contiguous shard (Philox keys are global env ids)."""
    return rank * envs_per_rank


@dataclass
class PPOConfig:
    n_envs: int = 4096
    n_steps: int = 64
    gamma: float = 0.99
    gae_lambda: float = 0.95
    clip_range: float = 0.2
    ent_coef: float = 0.0
    vf_coef: float = 0.5
    max_grad_norm: float = 0.5
    learning_rate: float = 3e-4  # train_hover.py:56
    n_epochs: int = 10
    batch_size: int = 8192
    norm_obs: bool = True  # train_hover.py:43
    norm_reward: bool = True
    clip_obs: float = 10.0
    clip_reward: float = 10.0
    seed: int = 0
    use_cuda_graph: bool = True
    target_kl: float = 0.0  # SB3 PPO target_kl: stop the epoch loop once the approximate KL exceeds 1.5 x this (0 = off)
    log_std_init: float = 0.0  # SB3 policy_kwargs log_std_init
    graph_update: bool = True  # replay captured optimiser steps instead of eager launches
    tf32_update: bool = True  # (fused_update=False only) library GEMMs of the torch update in TF32
    lr_final_frac: float = 1.0  # linear learning-rate schedule (SB3 lr callable): lr * (1 - (1 - lr_final_frac) * progress), progress from
    lr_anneal_iters: int = 0    # iteration / lr_anneal_iters clipped to 1 (0 = constant learning rate); fused update only
    recompute_old_logp: bool = False  # (fused update) old log-probs from the update kernel's own forward pass, see ppo_update_recompute_logp
    kl_stop_per_minibatch: bool = False  # target_kl checked per minibatch on the device (SB3) instead of on the epoch mean by the host
    log_std_min: float | None = None  # optional floor of log_std (fused update only): the exploration noise cannot collapse below exp(this)
    log_std_min_final: float | None = None  # ... released linearly to this value between the iterations log_std_min_iters = (start, end):
    log_std_min_iters: tuple = (0, 0)       # explore at a guaranteed noise level first, then let the policy narrow (0, 0 = constant floor)
    fused_update: bool = True  # the hand-written update kernels (ppo_update_*); False: torch autograd + torch.optim.Adam (reference)
    fuse_obs_stats: bool = False  # VecNormalize's obs statistics update inside the policy-forward launch (ppo_policy_forward_stats): one launch
                                  # fewer per env step, but measured SLOWER inside the two-branch rollout graph (3.30 vs 3.16 ms per 131 072 x 32
                                  # rollout): the in-kernel wait for the last CTA makes every CTA wait for the SMs the side branch still holds
    chain_obs_stats: bool = True  # the statistics launch and the policy-forward launch of a rollout step as programmatic dependents
                                  # (ppo_policy_forward_stats, fused = 0): hover 131 072 x 32: 3.14 -> 3.02 ms per rollout
    bootstrap_first: bool | None = None  # side branch: time-limit bootstrap before the reward normalisation (ppo_bootstrap_truncated_first +
                                         # ppo_reward_normalize_add).  None = where it measured faster: the yaw task, whose env step + reset are
                                         # shorter than the side branch (65 536 x 128 with the chain: 6.73 -> 6.06 ms; without either: 6.51 ms),
                                         # not the hover task (3.02 -> 3.07 ms)
    net_arch: int = HID  # hidden width of both MLPs: 128 = train_hover.py:57, 64 = SB3's default; < 128 runs zero-padded (ActorCritic)


class RolloutEngine:
    """``PPO.collect_rollouts`` with everything on the device: per env step

        VecNormalize obs statistics -> policy forward + sampling -> env step ->
        time-limit bootstrap -> env reset of finished episodes -> reward normalisation

    and GAE at the end.  The T-step loop is captured once into a CUDA graph and
    replayed, so a rollout costs one host call."""

    def __init__(self, sim: QuadXSim, policy: PackedPolicy, cfg: PPOConfig, row0: int = 0):
        self.sim, self.pol, self.cfg = sim, policy, cfg
        n, T, d = sim.n, cfg.n_steps, sim.device
        od, ad = sim.obs_dim, sim.act_dim
        self.n, self.T, self.device, self.row0 = n, T, d, row0
        f = dict(device=d, dtype=torch.float32)
        self.cur_obs = torch.zeros(n, od, **f)
        self.obs = torch.zeros(T, n, od, **f)  # normalised, as seen by the policy
        self.actions = torch.zeros(T, n, ad, **f)
        self.env_actions = torch.zeros(n, ad, **f)
        self.log_probs = torch.zeros(T, n, **f)
        self.values = torch.zeros(T, n, **f)
        self.rewards = torch.zeros(T, n, **f)
        self.raw_reward = torch.zeros(n, **f)
        self.dones = torch.zeros(T, n, dtype=torch.uint8, device=d)
        self.te = torch.zeros(n, dtype=torch.uint8, device=d)
        self.tr = torch.zeros(n, dtype=torch.uint8, device=d)
        self.terminal_obs = torch.zeros(n, od, **f)
        self.last_values = torch.zeros(n, **f)
        self.advantages = torch.zeros(T, n, **f)
        self.returns = torch.zeros(T, n, **f)
        self.returns_acc = torch.zeros(n, **f)
        self.obs_stats = RunningStats(od, d)
        self.ret_stats = RunningStats(1, d)
        self.step_base = torch.zeros(1, dtype=torch.int64, device=d)
        self._done_queue = sim.done_queue()
        self._graph = None
        self._side = torch.cuda.Stream(device=d)
        self._snap_mean = torch.zeros(2, od, **f)  # fp32 (mean, inv_std) of the observation statistics, one pair per step parity
        self._snap_inv = torch.ones(2, od, **f)
        self.sim.reset(self.cur_obs)
        # one-time kernel attribute setup must not happen inside a graph capture
        policy_forward(self.pol, self.cur_obs, deterministic=True, values=self.last_values)

    # one env step of the rollout, slot t.  Two streams (two branches of the captured graph):
    #   main: obs statistics -> policy forward + sampling -> env step -> reset of the finished envs        (the critical path)
    #   side: reward normalisation (return statistics) -> time-limit bootstrap                           (only GAE reads its results)
    # The side branch of step t reads what the env step wrote (raw reward, flags, terminal observations, the done queue) and the
    # observation statistics of step t, so (a) main joins it before the env step of t + 1 overwrites those, and (b) the fp32
    # (mean, inv_std) of step t live in the buffer pair t & 1, which the statistics update of step t + 1 does not touch.
    def _step(self, t: int) -> None:
        cfg, sim = self.cfg, self.sim
        stats = self.obs_stats if cfg.norm_obs else None
        norm = (self._snap_mean[t & 1], self._snap_inv[t & 1]) if cfg.norm_obs else None
        chain = cfg.norm_obs and (cfg.fuse_obs_stats or cfg.chain_obs_stats)
        if cfg.norm_obs and not chain:
            self.obs_stats.update(self.cur_obs, out=norm)
        policy_forward(self.pol, self.cur_obs, obs_stats=stats, norm=norm, obs_clip=cfg.clip_obs, seed=cfg.seed, row0=self.row0, step=t,
                       step_base=self.step_base, actions=self.actions[t], env_actions=self.env_actions, values=self.values[t],
                       log_probs=self.log_probs[t], obs_norm=self.obs[t], update_stats=chain, fused_stats=cfg.fuse_obs_stats)
        main = torch.cuda.current_stream(self.device)
        if t > 0:
            main.wait_stream(self._side)  # join the side branch of step t - 1 (the rollout ends with a join, so there is none at t = 0)
        sim.step_begin(self.env_actions, self.cur_obs, self.raw_reward, self.te, self.tr, self.terminal_obs)
        self._side.wait_stream(main)  # fork
        with torch.cuda.stream(self._side):
            boot_args = (self.pol, self.terminal_obs, norm, cfg.clip_obs, self._done_queue, self.te, self.tr, cfg.gamma, self.rewards[t])
            norm_args = (self.raw_reward, self.te, self.tr, self.returns_acc, self.ret_stats, cfg.gamma, cfg.clip_reward, self.rewards[t], self.dones[t])
            boot_first = cfg.bootstrap_first if cfg.bootstrap_first is not None else (sim.obs_dim != 20)  # yaw: 12-D observation
            if cfg.norm_reward and boot_first:
                # the bootstrap launch needs a whole SM's shared memory per CTA even to find the done queue empty: issued first it runs
                # while the main branch is still in the reset / statistics launches, not after the policy CTAs have taken the SMs
                bootstrap_truncated(*boot_args, first=True)
                reward_normalize(*norm_args, add=True)
            else:
                if cfg.norm_reward:
                    reward_normalize(*norm_args)
                else:
                    self.rewards[t].copy_(self.raw_reward)
                    torch.bitwise_or(self.te, self.tr, out=self.dones[t])
                # SB3: rewards[idx] += gamma * V(terminal_obs) when the time limit, not the task, ended the episode
                bootstrap_truncated(*boot_args)
        sim.step_end(self.cur_obs)

    def _rollout_body(self) -> None:
        for t in range(self.T):
            with torch.cuda.nvtx.range(f"rollout_step_{t}"):  # shows up per step in nsys / ncu timelines
                self._step(t)
        torch.cuda.current_stream(self.device).wait_stream(self._side)  # join: rewards / dones of the last step
        stats = self.obs_stats if self.cfg.norm_obs else None
        if stats is not None:  # the canonical fp32 copies (final forward, export, checkpoints) follow the last step's pair
            stats.mean.copy_(self._snap_mean[(self.T - 1) & 1]); stats.inv_std.copy_(self._snap_inv[(self.T - 1) & 1])
        policy_forward(self.pol, self.cur_obs, obs_stats=stats, obs_clip=self.cfg.clip_obs, deterministic=True, values=self.last_values)
        gae(self.rewards, self.values, self.dones, self.last_values, self.cfg.gamma, self.cfg.gae_lambda, self.advantages, self.returns)
        self.step_base += self.T

    def collect(self) -> None:
        """Fill the rollout buffers with T x n transitions and their advantages / returns."""
        if not self.cfg.use_cuda_graph:
            self._rollout_body()
            return
        if self._graph is None:
            self._graph = _capture(self._rollout_body, self.device)
        self._graph.replay()

    @property
    def launches_per_rollout(self) -> int:
        per_step = (1 if self.cfg.norm_obs and not self.cfg.fuse_obs_stats else 0) + 1 + 2 + 1 + 2  # obs stats, forward, env step/reset, bootstrap, reward path
        return self.T * per_step + 3


def module_params_in_layout_order(model: ActorCritic) -> list:
    """The parameters in the order of the flat vector of include/ppo_b200.h (ppo_update_num_params)."""
    m = model
    return [m.pi1.weight, m.pi1.bias, m.pi2.weight, m.pi2.bias, m.mu.weight, m.mu.bias,
            m.vf1.weight, m.vf1.bias, m.vf2.weight, m.vf2.bias, m.v.weight, m.v.bias, m.log_std]


class FusedUpdater:
    """SB3 ``PPO.train`` on the hand-written kernels (K5): per optimiser step ``ppo_update_minibatch`` (minibatch
    statistics, forward + loss + backward on the tensor cores, gradient reduction), the gradient all-reduce when there is
    more than one rank, and ``ppo_update_adam`` (global-norm clip, Adam, bf16 re-pack for the rollout's forward kernel).

    The module's parameters become views of one flat fp32 buffer (``self.flat``), which is what the Adam kernel updates;
    minibatches are sets of 128-row tiles of the rollout buffers (a random permutation of the tiles per epoch)."""

    def __init__(self, model: ActorCritic, packed: PackedPolicy, cfg: "PPOConfig", device, world: int = 1):
        self.model, self.packed, self.cfg, self.device, self.world = model, packed, cfg, _lib.cuda_device(device), world
        self.lib = _lib.lib()
        od, ad = model.obs_dim, model.act_dim
        self.n_params = int(self.lib.ppo_update_num_params(od, ad))
        params = module_params_in_layout_order(model)
        assert sum(p.numel() for p in params) == self.n_params and len(params) == len(list(model.parameters()))
        with torch.no_grad():
            self.flat = torch.cat([p.detach().reshape(-1) for p in params]).contiguous()
            o = 0
            for p in params:
                p.data = self.flat[o:o + p.numel()].view_as(p)
                o += p.numel()
        f = dict(device=self.device, dtype=torch.float32)
        self.grad = torch.zeros(self.n_params + 4, **f)  # + the two early-stop slots (ppo_update_kl_stop), padded to 16 bytes
        self.exp_avg = torch.zeros(self.n_params, **f)
        self.exp_avg_sq = torch.zeros(self.n_params, **f)
        self.loss_stats = torch.zeros(8, **f)
        self.workspace = torch.zeros(int(self.lib.ppo_update_workspace_bytes(od, ad)) // 4 + 4, **f)  # zero-filled once
        self._all_tiles = torch.arange((cfg.n_steps * cfg.n_envs + 127) // 128, dtype=torch.int32, device=self.device)  # recompute_logp
        packed.refresh()

    def gradient(self, ro: "RolloutEngine", tiles: torch.Tensor, normalize_adv: bool = True) -> torch.Tensor:
        """Mean gradient of the PPO loss over the minibatch `tiles` (int32 device tensor of 128-row tile indices)."""
        cfg, N = self.cfg, ro.T * ro.n
        assert tiles.dtype == torch.int32 and tiles.device == self.device and tiles.is_contiguous()
        check(self.lib.ppo_update_minibatch(C.byref(self.packed.struct), ptr(ro.obs), ptr(ro.actions), ptr(ro.log_probs), ptr(ro.advantages),
                                            ptr(ro.returns), ptr(tiles), tiles.numel(), N, cfg.clip_range, cfg.vf_coef, cfg.ent_coef,
                                            int(normalize_adv), ptr(self.grad), ptr(self.loss_stats), ptr(self.workspace), stream(self.device)))
        return self.grad[:self.n_params]

    def apply(self) -> None:
        """All-reduce (world > 1), clip, Adam, re-pack."""
        cfg, s = self.cfg, stream(self.device)
        scale = 1.0
        if self.world > 1:
            dist.all_reduce(self.grad)
            scale = 1.0 / self.world
            check(self.lib.ppo_update_grad_norm(ptr(self.grad), self.n_params, scale, ptr(self.workspace), s))
        check(self.lib.ppo_update_adam(ptr(self.flat), ptr(self.grad), ptr(self.exp_avg), ptr(self.exp_avg_sq), self.n_params, cfg.learning_rate,
                                       0.9, 0.999, 1e-5, cfg.max_grad_norm, scale, C.byref(self.packed.struct), ptr(self.workspace), s))

    def step(self, ro: "RolloutEngine", tiles: torch.Tensor) -> None:
        self.gradient(ro, tiles)
        self.apply()

    def recompute_logp(self, ro: "RolloutEngine") -> None:
        """Overwrite the rollout's log-probs with the update kernel's own forward pass (ppo_update_recompute_logp)."""
        N, n_tiles = ro.T * ro.n, self._all_tiles.numel()
        assert (N + 127) // 128 == n_tiles, "the rollout is not the n_steps x n_envs of the updater's config"
        check(self.lib.ppo_update_recompute_logp(C.byref(self.packed.struct), ptr(ro.obs), ptr(ro.actions), ptr(self._all_tiles), n_tiles, N,
                                                 ptr(ro.log_probs), ptr(self.workspace), stream(self.device)))

    def arm_kl_stop(self, target_kl: float) -> None:
        """(Re-)arm SB3's target_kl early stop on the device (0 = off) and clear its latch: call once per PPO.train."""
        check(self.lib.ppo_update_kl_stop(ptr(self.workspace), float(target_kl), None, None, stream(self.device)))

    def kl_stopped(self) -> tuple[bool, int]:
        """(latched, optimiser steps skipped since arm_kl_stop)."""
        st, sk = C.c_int32(), C.c_int32()
        check(self.lib.ppo_update_kl_stop(ptr(self.workspace), -1.0, C.byref(st), C.byref(sk), stream(self.device)))
        return bool(st.value), sk.value

    def set_log_std_floor(self, floor: float | None) -> None:
        check(self.lib.ppo_update_set_log_std_floor(ptr(self.workspace), 0 if floor is None else 1, 0.0 if floor is None else float(floor), stream(self.device)))

    def set_lr_scale(self, scale: float) -> None:
        """Learning-rate schedule: later optimiser steps (graph replays included) use learning_rate * scale."""
        check(self.lib.ppo_update_set_lr_scale(ptr(self.workspace), float(scale), stream(self.device)))

    @property
    def adam_steps(self) -> int:
        out = C.c_int64()
        check(self.lib.ppo_update_step_count(ptr(self.workspace), -1, C.byref(out), stream(self.device)))
        return out.value

    def state_dict(self) -> dict:
        return {"flat": self.flat.clone(), "exp_avg": self.exp_avg.clone(), "exp_avg_sq": self.exp_avg_sq.clone(), "adam_steps": self.adam_steps}

    def load_state_dict(self, sd: dict) -> None:
        self.flat.copy_(sd["flat"]); self.exp_avg.copy_(sd["exp_avg"]); self.exp_avg_sq.copy_(sd["exp_avg_sq"])
        check(self.lib.ppo_update_step_count(ptr(self.workspace), int(sd["adam_steps"]), None, stream(self.device)))
        self.packed.refresh()


class PPOTrainer:
    """``PPO.learn`` (train_hover.py:47-60, with PPO instead of SAC as the north star asks)."""

    def __init__(self, cfg: PPOConfig, device=None, env_cfg=None, rank: int = 0, world: int = 1, task: int = 0):
        """task: QX_TASK_HOVER (0, hover.py) or QX_TASK_YAW (1, yaw.py: 12-D obs, 1-D action)."""
        self.cfg, self.rank, self.world = cfg, rank, world
        self.device = dev = _lib.cuda_device(device)
        if cfg.tf32_update:
            torch.backends.cuda.matmul.allow_tf32 = True
        torch.manual_seed(cfg.seed)  # identical initial weights on every rank
        self.model = (ActorCritic(log_std_init=cfg.log_std_init, hidden=cfg.net_arch) if task == 0
                      else ActorCritic(12, 1, log_std_init=cfg.log_std_init, hidden=cfg.net_arch)).to(dev)
        self.packed = PackedPolicy(self.model, dev)
        ecfg = env_cfg if env_cfg is not None else default_config(task)
        ecfg.update(auto_reset=1)
        self.sim = QuadXSim(cfg.n_envs, ecfg, seed=cfg.seed, env_id0=shard_env_ids(rank, cfg.n_envs), device=dev, task=task)
        self.rollout = RolloutEngine(self.sim, self.packed, cfg, row0=shard_env_ids(rank, cfg.n_envs))
        self.fused = FusedUpdater(self.model, self.packed, cfg, dev, world) if cfg.fused_update else None
        if self.fused is not None and cfg.log_std_min is not None:
            self.fused.set_log_std_floor(cfg.log_std_min)
        self.opt = None if cfg.fused_update else torch.optim.Adam(self.model.parameters(), lr=cfg.learning_rate, eps=1e-5,
                                                                   capturable=bool(cfg.graph_update and world == 1))
        self._epoch_graph = None
        self._update_graph = None  # (fused_update=False) one torch minibatch step, see _build_update_graph
        self._perm = torch.zeros_like(self.fused._all_tiles) if self.fused is not None else None  # the epoch's permutation of the tiles
        self.num_timesteps = 0
        self._iteration = 0
        self._evaluator = None  # PolicyEvaluator of evaluate(), built on its first call
        self.gen = torch.Generator(device=dev).manual_seed(cfg.seed + 1000 + rank)

    # one PPO minibatch: loss of SB3's PPO.train (clipped surrogate + vf_coef * MSE - ent_coef * entropy, advantages
    # normalised per minibatch) and the diagnostics it logs; `acc` accumulates [pg, vf, kl, clipfrac, approx_kl_k3]
    def _minibatch_loss(self, idx: torch.Tensor, acc: torch.Tensor) -> torch.Tensor:
        cfg, ro = self.cfg, self.rollout
        N = ro.T * ro.n
        obs, act = ro.obs.view(N, -1), ro.actions.view(N, -1)
        old_logp, adv_all, ret_all = ro.log_probs.view(N), ro.advantages.view(N), ro.returns.view(N)
        adv = adv_all[idx]
        adv = (adv - adv.mean()) / (adv.std() + 1e-8)
        value, logp, entropy = self.model.evaluate_actions(obs[idx], act[idx])
        lr_ = logp - old_logp[idx]
        ratio = torch.exp(lr_)
        pg = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 1 - cfg.clip_range, 1 + cfg.clip_range)).mean()
        vf = torch.nn.functional.mse_loss(ret_all[idx], value)
        loss = pg + cfg.vf_coef * vf - cfg.ent_coef * entropy.mean()
        with torch.no_grad():
            acc += torch.stack([pg.detach(), vf.detach(), -lr_.mean(), ((ratio - 1).abs() > cfg.clip_range).float().mean(),
                                ((ratio - 1) - lr_).mean()])
        return loss

    def _step_eager(self, idx: torch.Tensor, acc: torch.Tensor) -> None:
        loss = self._minibatch_loss(idx, acc)
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        allreduce_gradients(self.model.parameters(), self.world)
        torch.nn.utils.clip_grad_norm_(self.model.parameters(), self.cfg.max_grad_norm)
        self.opt.step()

    def _build_update_graph(self, bs: int) -> None:
        """(fused_update=False) Capture one torch minibatch step (gather, forward, loss, backward, grad clip, Adam) into a
        CUDA graph.  Single-GPU only.  The optimiser state tensors the graph updates are the ones the warm-up created:
        they are restored IN PLACE afterwards (Optimizer.load_state_dict would replace them and orphan the graph's)."""
        self._g_idx = torch.zeros(bs, dtype=torch.int64, device=self.device)
        self._g_acc = torch.zeros(5, device=self.device)
        if not self.opt.state:  # create the state tensors with one eager step, so that there is something to snapshot
            self._step_eager(self._g_idx, self._g_acc)
            for st in self.opt.state.values():
                for v in st.values():
                    if torch.is_tensor(v):
                        v.zero_()
        model_sd = {k: v.clone() for k, v in self.model.state_dict().items()}
        opt_snap = [{k: v.clone() for k, v in st.items() if torch.is_tensor(v)} for st in self.opt.state.values()]
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for _ in range(3):  # warm-up on a side stream, as CUDA-graph capture of an optimiser requires
                self._step_eager(self._g_idx, self._g_acc)
        torch.cuda.current_stream(self.device).wait_stream(side)
        self.opt.zero_grad(set_to_none=True)
        self._update_graph = _capture(lambda: self._step_eager(self._g_idx, self._g_acc), self.device)
        with torch.no_grad():  # the warm-up / capture steps must not count as training
            for k, v in self.model.state_dict().items():
                v.copy_(model_sd[k])
            for st, snap in zip(self.opt.state.values(), opt_snap):
                for k, v in snap.items():
                    st[k].copy_(v)

    def _update_fused(self) -> dict:
        """SB3 PPO.train on the hand-written kernels: per epoch a fresh random permutation of the rollout's 128-row tiles,
        cut into minibatches of batch_size rows; the optimiser steps of one epoch are one CUDA-graph replay (kernels and,
        with several ranks, the gradient all-reduce)."""
        cfg, ro, fu = self.cfg, self.rollout, self.fused
        N = ro.T * ro.n
        n_tiles = (N + 127) // 128
        tpm = max(1, min(cfg.batch_size, N) // 128)  # tiles per minibatch
        starts = list(range(0, n_tiles - tpm + 1, tpm)) or [0]

        def epoch_body():
            for s0 in starts:
                fu.step(ro, self._perm[s0:s0 + min(tpm, n_tiles - s0)])

        fu.loss_stats.zero_()
        if cfg.recompute_old_logp:
            fu.recompute_logp(ro)
        dev_kl = cfg.target_kl if cfg.kl_stop_per_minibatch else 0.0
        fu.arm_kl_stop(dev_kl)
        steps_before = fu.adam_steps
        for _ in range(cfg.n_epochs):
            self._perm.copy_(torch.randperm(n_tiles, device=self.device, generator=self.gen).to(torch.int32))
            kl_before, n_before = (float(fu.loss_stats[4]), float(fu.loss_stats[5])) if cfg.target_kl > 0.0 and not cfg.kl_stop_per_minibatch else (0.0, 0.0)
            if cfg.graph_update:
                if self._epoch_graph is None:
                    keep = {k: v.clone() for k, v in fu.state_dict().items() if torch.is_tensor(v)}
                    steps0, stats0 = fu.adam_steps, fu.loss_stats.clone()
                    side = torch.cuda.Stream(device=self.device)
                    side.wait_stream(torch.cuda.current_stream(self.device))
                    with torch.cuda.stream(side):
                        fu.step(ro, self._perm[:tpm])  # warm-up outside capture (one-time kernel attributes, NCCL)
                    torch.cuda.current_stream(self.device).wait_stream(side)
                    torch.cuda.synchronize(self.device)
                    self._epoch_graph = _capture(epoch_body, self.device)
                    # warm-up and capture must not count as training: restore parameters, moments, step count, statistics
                    fu.load_state_dict({**keep, "adam_steps": steps0})
                    fu.loss_stats.copy_(stats0)
                    fu.arm_kl_stop(dev_kl)
                self._epoch_graph.replay()
            else:
                epoch_body()
            if cfg.target_kl > 0.0 and cfg.kl_stop_per_minibatch:
                # the stop is taken on the device, per minibatch and identically on every rank (ppo_update_kl_stop); the host only
                # looks at the latch once per epoch to save itself the launches of the remaining epochs
                if fu.kl_stopped()[0]:
                    break
            elif cfg.target_kl > 0.0:  # epoch mean of the approximate KL, one host sync per epoch
                akl = torch.tensor([(float(fu.loss_stats[4]) - kl_before) / max(float(fu.loss_stats[5]) - n_before, 1.0)], device=self.device)
                if self.world > 1:
                    dist.all_reduce(akl)
                    akl /= self.world
                if float(akl) > 1.5 * cfg.target_kl:
                    break
        st = fu.loss_stats.tolist()
        n = max(st[5], 1.0)
        return {"pg": st[0] / n, "vf": st[1] / n, "kl": st[2] / n, "clipfrac": st[3] / n, "optimizer_steps": fu.adam_steps - steps_before}

    def update(self) -> dict:
        """SB3 PPO.train: n_epochs passes over the rollout in shuffled minibatches; target_kl ends the training of this rollout
        once the approximate KL exceeds 1.5 x target: on the mean of an epoch (one host sync per epoch; the default -- measured
        to learn faster on this task) or, with kl_stop_per_minibatch, at the first minibatch over the threshold and before its
        optimiser step as SB3 does, decided on the device (ppo_update_kl_stop)."""
        if self.fused is not None:
            return self._update_fused()
        cfg, ro = self.cfg, self.rollout
        N = ro.T * ro.n
        bs = min(cfg.batch_size, N)
        use_graph = cfg.graph_update and self.world == 1
        if use_graph and self._update_graph is None:
            self._build_update_graph(bs)
        acc = self._g_acc if use_graph else torch.zeros(5, device=self.device)
        acc.zero_()
        n_mb = 0
        for _ in range(cfg.n_epochs):
            perm = torch.randperm(N, device=self.device, generator=self.gen)
            kl_before = acc[4].clone()
            n_epoch = 0
            for s in range(0, N - bs + 1, bs):
                if use_graph:
                    self._g_idx.copy_(perm[s:s + bs])
                    self._update_graph.replay()
                else:
                    self._step_eager(perm[s:s + bs], acc)
                n_epoch += 1
            n_mb += n_epoch
            if cfg.target_kl > 0.0:
                akl = (acc[4] - kl_before) / max(n_epoch, 1)
                if self.world > 1:
                    dist.all_reduce(akl)
                    akl /= self.world
                if float(akl) > 1.5 * cfg.target_kl:
                    break
        self.packed.refresh()
        out = (acc / max(n_mb, 1)).tolist()
        return {"pg": out[0], "vf": out[1], "kl": out[2], "clipfrac": out[3]}

    def learn_iteration(self) -> dict:
        if self.fused is not None and self.cfg.lr_anneal_iters > 0:
            prog = min(1.0, self._iteration / self.cfg.lr_anneal_iters)
            self.fused.set_lr_scale(1.0 - (1.0 - self.cfg.lr_final_frac) * prog)
        if self.fused is not None and self.cfg.log_std_min is not None and self.cfg.log_std_min_final is not None:
            a, b = self.cfg.log_std_min_iters
            prog = 0.0 if self._iteration <= a else (1.0 if b <= a or self._iteration >= b else (self._iteration - a) / (b - a))
            self.fused.set_log_std_floor(self.cfg.log_std_min + (self.cfg.log_std_min_final - self.cfg.log_std_min) * prog)
        self._iteration += 1
        with torch.cuda.nvtx.range("ppo_collect_rollouts"):
            self.rollout.collect()
        self.num_timesteps += self.rollout.T * self.rollout.n * self.world
        if self.world > 1:  # every rank normalises with the statistics of all shards (outside the captured rollout graph)
            self.rollout.obs_stats.allreduce_()
            self.rollout.ret_stats.allreduce_()
        with torch.cuda.nvtx.range("ppo_update"):
            out = self.update()
        s, l, c = self.sim.episode_stats(clear=True)
        if self.world > 1:
            t = torch.tensor([s, float(l), float(c)], device=self.device, dtype=torch.float64)
            dist.all_reduce(t)
            s, l, c = float(t[0]), float(t[1]), float(t[2])
        out.update(ep_rew_mean=s / c if c else float("nan"), ep_len_mean=l / c if c else float("nan"), episodes=int(c),
                   timesteps=self.num_timesteps)
        return out

    def evaluate(self, n_episodes: int = 4096, seed: int | None = None) -> tuple[dict, dict]:
        """EvalCallback's evaluation of the current policy: PolicyEvaluator on the trainer's packed weights, its VecNormalize
        observation statistics (frozen for the evaluation), clip_obs, task and env config; seed None = cfg.seed + 1.  The
        evaluator (its own sim and graph) is built on the first call and kept while (n_episodes, seed) stay the same.  Reads the
        policy and the statistics only: no rollout buffer, statistic, random stream or env of training changes."""
        seed = self.cfg.seed + 1 if seed is None else int(seed)
        ev = self._evaluator
        if ev is None or (ev.n, ev.seed) != (n_episodes, seed):
            if ev is not None:
                ev.close()
            ev = PolicyEvaluator(self.packed, self.rollout.obs_stats if self.cfg.norm_obs else None, self.sim.cfg, n_episodes, seed,
                                 task=self.sim.cfg.task, obs_clip=self.cfg.clip_obs, device=self.device)
            self._evaluator = ev
        return ev.evaluate()

    def save(self, path: str) -> None:
        """Counterpart of model.save + env.save (train_hover.py:26-27,62-63): policy, optimiser, VecNormalize statistics, and
        what a resumed run needs to continue the same random streams (sampling counter, return accumulator, minibatch RNG)."""
        opt = self.fused.state_dict() if self.fused is not None else self.opt.state_dict()
        torch.save({"model": self.model.state_dict(), "opt": opt, "fused": self.fused is not None,
                    "obs_stats": self.rollout.obs_stats.state_dict(), "ret_stats": self.rollout.ret_stats.state_dict(),
                    "num_timesteps": self.num_timesteps, "cfg": dict(self.cfg.__dict__),
                    "step_base": self.rollout.step_base.clone(), "returns_acc": self.rollout.returns_acc.clone(), "gen_state": self.gen.get_state(),
                    "sb3_policy_state_dict": export_sb3_state_dict(self.model),
                    "sb3_vecnormalize": {k: (torch.as_tensor(v) if not isinstance(v, dict) else {kk: torch.as_tensor(vv) for kk, vv in v.items()})
                                         for k, v in export_vecnormalize(self.rollout.obs_stats, self.rollout.ret_stats, self.cfg).items()}}, path)

    def save_sb3(self, path: str) -> None:
        """The policy as an SB3-style archive (policy.pth + version + VecNormalize statistics), see export_sb3_zip."""
        c = self.cfg
        hyper = dict(log_std_init=c.log_std_init, learning_rate=c.learning_rate, n_steps=c.n_steps, batch_size=c.batch_size, gamma=c.gamma,
                     gae_lambda=c.gae_lambda, clip_range=c.clip_range, ent_coef=c.ent_coef, vf_coef=c.vf_coef, max_grad_norm=c.max_grad_norm,
                     num_timesteps=int(self.num_timesteps))
        export_sb3_zip(self.model, path, export_vecnormalize(self.rollout.obs_stats, self.rollout.ret_stats, self.cfg), hyper=hyper)

    def load(self, path: str) -> None:
        sd = torch.load(path, map_location=self.device, weights_only=True)  # tensors and plain containers only: no pickle execution
        if bool(sd.get("fused", False)) != (self.fused is not None):
            raise ValueError("checkpoint was written with a different PPOConfig.fused_update")
        with torch.no_grad():  # in place: the parameters are views of the flat buffer / captured by CUDA graphs
            for k, v in self.model.state_dict().items():
                v.copy_(sd["model"][k])
        if self.fused is not None:
            self.fused.load_state_dict(sd["opt"])
        else:
            if self._update_graph is not None and self.opt.state:
                for st, src in zip(self.opt.state.values(), sd["opt"]["state"].values()):  # in place: the graph updates these tensors
                    for k, v in src.items():
                        if torch.is_tensor(v):
                            st[k].copy_(v)
            else:
                self.opt.load_state_dict(sd["opt"])
        self.rollout.obs_stats.load_state_dict(sd["obs_stats"]); self.rollout.ret_stats.load_state_dict(sd["ret_stats"])
        self.rollout.step_base.copy_(sd["step_base"]); self.rollout.returns_acc.copy_(sd["returns_acc"])
        self.gen.set_state(sd["gen_state"].cpu())
        self.num_timesteps = int(sd["num_timesteps"])
        self.packed.refresh()
