"""Play back stable-baselines3 checkpoints on the device: the reference trains SAC (train_hover.py:47-58,
``SAC("MlpPolicy", policy_kwargs=dict(net_arch=[128, 128]))``) and plays the ``.zip`` + VecNormalize pair back with
``model.predict(obs, deterministic=True)`` (test_hover.py:7-27).

- ``SacActor``: SB3's ``Actor`` under its parameter names (``latent_pi.0``, ``latent_pi.2``, ``mu``, ``log_std``) with a torch
  forward of the deterministic action, ``tanh(mu(relu(relu(x))))`` -- the reference the kernel is tested against.
- ``PackedSacActor`` / ``sac_actor_forward``: the bf16 layout of ``struct SacActor`` and the tcgen05 kernel K8 of
  include/sac_b200.h (VecNormalize + actor in one launch).
- ``load_sb3_zip``: reads an SB3 model archive with ``zipfile`` and ``torch.load(weights_only=True)`` -- SB3 is not needed
  and nothing is unpickled.  SAC archives give a ``SacActor``; PPO archives (SB3's own or ``ppo.export_sb3_zip``'s) an
  ``ActorCritic``.  Whatever the kernels cannot run exactly is refused with the reason.
- ``load_vecnormalize`` / ``obs_stats_from_vecnormalize``: VecNormalize statistics in the ``.npz`` form of
  ``ppo.export_sb3_zip`` (tools/sb3_vecnormalize_to_npz.py converts SB3's ``.pkl`` on the reference side).

SAC training (replay buffer, twin critics, the update) is not here; only the actor's deterministic action is.
"""
from __future__ import annotations

import ctypes as C
import io
import json
import zipfile
from dataclasses import dataclass

import numpy as np
import torch
from torch import nn

from . import _lib
from ._lib import SacActor as SacActorStruct
from ._lib import check, expect, ptr, stream
from .ppo import ActorCritic, PackedPolicy, RunningStats, import_sb3_state_dict

HID, IN_PAD, HEAD_PAD = 128, 32, 16  # SAC_HIDDEN, SAC_IN_PAD, SAC_HEAD_PAD of include/sac_b200.h


class SacActor(nn.Module):
    """SB3 ``Actor`` of ``SACPolicy`` (``MlpPolicy``, ReLU, no gSDE): ``latent_pi`` = Linear-ReLU-Linear-ReLU, ``mu`` and the
    state-dependent ``log_std`` head.  ``forward`` is the deterministic action ``tanh(mu(latent_pi(obs)))`` (the mode of
    SquashedDiagGaussianDistribution); ``log_std`` is carried so that an archive's actor loads whole, and is not used."""

    def __init__(self, obs_dim: int = 20, act_dim: int = 4, net_arch: tuple = (HID, HID)):
        super().__init__()
        h1, h2 = net_arch
        self.obs_dim, self.act_dim, self.net_arch = obs_dim, act_dim, (int(h1), int(h2))
        self.latent_pi = nn.Sequential(nn.Linear(obs_dim, h1), nn.ReLU(), nn.Linear(h1, h2), nn.ReLU())
        self.mu = nn.Linear(h2, act_dim)
        self.log_std = nn.Linear(h2, act_dim)

    def forward(self, obs: torch.Tensor) -> torch.Tensor:
        return torch.tanh(self.mu(self.latent_pi(obs)))


class PackedSacActor:
    """bf16 copy of a ``SacActor`` in the layout of ``struct SacActor`` (hidden widths < 128 zero-padded: a padded unit
    computes relu(0) = 0 and feeds nothing downstream)."""

    def __init__(self, actor: SacActor, device):
        if actor.obs_dim > IN_PAD or actor.act_dim > 4 or max(actor.net_arch) > HID:
            raise ValueError(f"SacActor obs_dim {actor.obs_dim}, act_dim {actor.act_dim}, net_arch {actor.net_arch}: the kernel takes "
                             f"obs_dim <= {IN_PAD}, act_dim <= 4 and widths <= {HID}")
        self.model, self.device = actor, _lib.cuda_device(device)
        d = self.device
        self.w1 = torch.zeros(HID, IN_PAD, dtype=torch.bfloat16, device=d)
        self.w2 = torch.zeros(HID, HID, dtype=torch.bfloat16, device=d)
        self.w_mu = torch.zeros(HEAD_PAD, HID, dtype=torch.bfloat16, device=d)
        self.b1 = torch.zeros(HID, device=d)
        self.b2 = torch.zeros(HID, device=d)
        self.b_mu = torch.zeros(HEAD_PAD, device=d)
        self.struct = SacActorStruct(self.w1.data_ptr(), self.w2.data_ptr(), self.w_mu.data_ptr(), self.b1.data_ptr(), self.b2.data_ptr(),
                                     self.b_mu.data_ptr(), actor.obs_dim, actor.act_dim)
        self.refresh()

    @torch.no_grad()
    def refresh(self) -> None:
        """Re-pack after the actor's weights changed."""
        l1, l2, mu = self.model.latent_pi[0], self.model.latent_pi[2], self.model.mu
        h1, h2 = self.model.net_arch
        od, ad = self.model.obs_dim, self.model.act_dim
        self.w1[:h1, :od].copy_(l1.weight)
        self.w2[:h2, :h1].copy_(l2.weight)
        self.w_mu[:ad, :h2].copy_(mu.weight)
        self.b1[:h1].copy_(l1.bias)
        self.b2[:h2].copy_(l2.bias)
        self.b_mu[:ad].copy_(mu.bias)

    def act(self, obs: torch.Tensor, env_actions: torch.Tensor, norm: tuple | None, obs_clip: float) -> None:
        """The deterministic action of one playback step (``SAC.predict(obs, deterministic=True)``) into env_actions: tanh
        keeps it in [-1, 1], the action box of both tasks, so SB3's unscale_action is the identity.  The counterpart of
        ``ppo.PackedPolicy.act``, so that ``ppo.PolicyEvaluator`` serves both."""
        sac_actor_forward(self, obs, norm=norm, obs_clip=obs_clip, actions=env_actions)


def sac_actor_forward(actor: PackedSacActor, obs: torch.Tensor, *, actions: torch.Tensor, norm: tuple | None = None, obs_clip: float = 10.0,
                      obs_norm: torch.Tensor | None = None) -> None:
    """VecNormalize.normalize_obs (with norm = (mean, inv_std); obs_clip <= 0: no clip) + SB3 Actor deterministic forward on the
    tensor cores (sac_actor_forward, K8): actions [n, act_dim], obs_norm [n, obs_dim] (optional, the normalised input)."""
    n, dev = obs.shape[0], actor.device
    od, ad = actor.model.obs_dim, actor.model.act_dim
    if obs.dim() != 2 or obs.shape[1] != od or obs.dtype != torch.float32 or obs.device != dev or obs.stride(1) != 1:
        raise ValueError(f"obs: expected [n, {od}] float32 rows with unit column stride on {dev}; got {obs.dtype} {tuple(obs.shape)} "
                         f"strides {obs.stride()} on {obs.device}")
    expect(actions, "actions", dtype=torch.float32, device=dev, numel=n * ad)
    if obs_norm is not None:
        expect(obs_norm, "obs_norm", dtype=torch.float32, device=dev, numel=n * od)
    mean, inv_std = norm if norm is not None else (None, None)
    for name, t in (("mean", mean), ("inv_std", inv_std)):
        if t is not None:
            expect(t, name, dtype=torch.float32, device=dev, numel=od)
    check(_lib.lib().sac_actor_forward(C.byref(actor.struct), ptr(obs), obs.stride(0), n, ptr(mean), ptr(inv_std), obs_clip, ptr(actions),
                                       ptr(obs_norm), stream(dev)))


# ------------------------------------------------------------------------------------------------------------------------------
# stable-baselines3 archives
# ------------------------------------------------------------------------------------------------------------------------------
_RELU = {"torch.nn.ReLU", "torch.nn.modules.activation.ReLU", "ReLU", "<class 'torch.nn.modules.activation.ReLU'>"}
_TANH = {"torch.nn.Tanh", "torch.nn.modules.activation.Tanh", "Tanh", "<class 'torch.nn.modules.activation.Tanh'>"}


@dataclass
class Sb3Archive:
    """What ``load_sb3_zip`` read: ``algorithm`` "SAC" or "PPO", ``model`` (``SacActor`` / ``ppo.ActorCritic``), the
    archive's own VecNormalize statistics (``vecnormalize.npz``, written by ``ppo.export_sb3_zip``) if it has them, and the
    SB3 version it names."""

    algorithm: str
    model: nn.Module
    vecnormalize: dict | None
    sb3_version: str | None

    def pack(self, device) -> "PackedSacActor | PackedPolicy":
        """The packed policy the kernels run (``ppo.PolicyEvaluator`` / ``ppo.evaluate_policy`` take either)."""
        return PackedSacActor(self.model, device) if self.algorithm == "SAC" else PackedPolicy(self.model, device)


def _hidden_layers(sd: dict, prefix: str, path: str) -> list:
    """The (weight, bias) pairs of an SB3 MLP `prefix`.0, .2, ...: exactly two, each at most HID wide."""
    idx = sorted(int(k[len(prefix) + 1:].split(".")[0]) for k in sd if k.startswith(prefix + ".") and k.endswith(".weight"))
    if idx != [0, 2]:
        raise ValueError(f"{path}: {prefix} has {len(idx)} linear layers ({[f'{prefix}.{i}' for i in idx]}); the kernels run exactly two "
                         f"hidden layers (net_arch=[h1, h2])")
    layers = [(sd[f"{prefix}.{i}.weight"], sd[f"{prefix}.{i}.bias"]) for i in idx]
    for i, (w, _) in zip(idx, layers):
        if w.shape[0] > HID:
            raise ValueError(f"{path}: {prefix}.{i} is {w.shape[0]} units wide; hidden widths above {HID} are not supported")
    return layers


def _activation(data: dict, default: str, allowed: set, algo: str, path: str) -> None:
    kw = data.get("policy_kwargs", {})
    if isinstance(kw, dict) and ":serialized:" in kw:
        raise ValueError(f"{path}: policy_kwargs is stored as a cloudpickle (it holds a Python object, e.g. an activation_fn class); "
                         f"reading it would mean unpickling arbitrary code, which this loader does not do")
    if not isinstance(kw, dict):
        raise ValueError(f"{path}: policy_kwargs is not a plain mapping: {kw!r}")
    act = kw.get("activation_fn", default)
    if str(act) not in allowed:
        raise ValueError(f"{path}: {algo} activation_fn {act!r} is not supported: the {algo} kernel runs {default} only")


def load_sb3_zip(path: str, device="cpu") -> Sb3Archive:
    """Read a stable-baselines3 model archive (``model.save`` / ``CheckpointCallback``: members ``data``, ``policy.pth``, ...)
    without SB3 and without unpickling: ``data`` is read as JSON, ``policy.pth`` with ``torch.load(weights_only=True)``.

    SAC is recognised by the ``actor.latent_pi.*`` keys; only ``actor.*`` is used (critics and optimisers are ignored), the
    activation is ReLU unless ``policy_kwargs`` names another.  PPO is recognised by ``mlp_extractor.*`` / ``action_net``
    and must be Tanh (SB3's default; K2 is tanh-only).  Refused, each with its reason: a cloudpickled ``policy_kwargs``,
    another activation, widths above 128, other than two hidden layers, gSDE, obs_dim > 32, act_dim > 4."""
    with zipfile.ZipFile(path) as z:
        names = set(z.namelist())
        if "policy.pth" not in names:
            raise ValueError(f"{path}: no policy.pth member; not a stable-baselines3 model archive")
        data = json.loads(z.read("data").decode()) if "data" in names else {}
        sd = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
        version = z.read("_stable_baselines3_version").decode().strip() if "_stable_baselines3_version" in names else None
        vn = _read_npz(z.read("vecnormalize.npz")) if "vecnormalize.npz" in names else None
    kw = data.get("policy_kwargs", {})
    if data.get("use_sde", False) or (isinstance(kw, dict) and kw.get("use_sde", False)):
        raise ValueError(f"{path}: the policy was trained with gSDE (use_sde=True); gSDE is not supported")
    if any(k.startswith("actor.latent_pi.") for k in sd):
        if "actor.log_std" in sd:
            raise ValueError(f"{path}: the actor carries a gSDE log_std matrix; gSDE is not supported")
        _activation(data, "ReLU", _RELU, "SAC", path)
        (w1, b1), (w2, b2) = _hidden_layers(sd, "actor.latent_pi", path)
        w_mu, b_mu = sd["actor.mu.weight"], sd["actor.mu.bias"]
        od, ad = int(w1.shape[1]), int(w_mu.shape[0])
        _check_dims(od, ad, path)
        model = SacActor(od, ad, (int(w1.shape[0]), int(w2.shape[0])))
        model.load_state_dict({k[len("actor."):]: v for k, v in sd.items() if k.startswith("actor.") and not k.startswith("actor.features_extractor.")})
        return Sb3Archive("SAC", model.to(device), vn, version)
    if any(k.startswith("mlp_extractor.") for k in sd) and "action_net.weight" in sd:
        if "log_std" in sd and sd["log_std"].dim() != 1:
            raise ValueError(f"{path}: the policy carries a gSDE log_std matrix; gSDE is not supported")
        _activation(data, "Tanh", _TANH, "PPO", path)
        (w1, _), (w2, _) = _hidden_layers(sd, "mlp_extractor.policy_net", path)
        _hidden_layers(sd, "mlp_extractor.value_net", path)
        od, ad = int(w1.shape[1]), int(sd["action_net.weight"].shape[0])
        _check_dims(od, ad, path)
        model = ActorCritic(od, ad, hidden=int(w1.shape[0]))
        import_sb3_state_dict(model, sd)
        return Sb3Archive("PPO", model.to(device), vn, version)
    raise ValueError(f"{path}: policy.pth has neither SAC actor keys (actor.latent_pi.*) nor PPO keys (mlp_extractor.*, action_net.*)")


def _check_dims(od: int, ad: int, path: str) -> None:
    if od > IN_PAD:
        raise ValueError(f"{path}: observation width {od} > {IN_PAD} is not supported")
    if ad > 4:
        raise ValueError(f"{path}: action width {ad} > 4 is not supported")


def _read_npz(raw: bytes) -> dict:
    with np.load(io.BytesIO(raw), allow_pickle=False) as f:
        return {k: f[k] for k in f.files}


def load_vecnormalize(path: str) -> dict:
    """VecNormalize statistics from an ``.npz`` with the keys ``ppo.export_sb3_zip`` writes (``obs_rms.mean``, ``obs_rms.var``,
    ``obs_rms.count``, ``clip_obs``, ``epsilon``, ``norm_obs``, ...); no pickles."""
    with open(path, "rb") as f:
        return _read_npz(f.read())


def obs_stats_from_vecnormalize(vn: dict, device) -> RunningStats | None:
    """The observation statistics as the device keeps them (``ppo.RunningStats``), None when ``norm_obs`` is off.  The fp32
    (mean, inv_std) are computed as the statistics kernels compute them: mean cast from fp64, inv_std = 1 / sqrt(var + eps)
    in fp64 with eps rounded to fp32 first, then cast."""
    if "norm_obs" in vn and not bool(vn["norm_obs"]):
        return None
    mean, var = np.asarray(vn["obs_rms.mean"], np.float64), np.asarray(vn["obs_rms.var"], np.float64)
    count, eps = float(vn["obs_rms.count"]), float(np.float32(vn.get("epsilon", 1e-8)))
    st = RunningStats(mean.size, device, eps=float(vn.get("epsilon", 1e-8)))
    st.stats.copy_(torch.from_numpy(np.concatenate([mean, var, [count]])))
    st.mean.copy_(torch.from_numpy(mean.astype(np.float32)))
    st.inv_std.copy_(torch.from_numpy((1.0 / np.sqrt(var + eps)).astype(np.float32)))
    return st
