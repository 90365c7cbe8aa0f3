"""CPU: reading stable-baselines3 model archives (sac.load_sb3_zip) and the SAC actor's torch forward.

The archives are built here with SB3's real member names (``data``, ``policy.pth``, ``actor.optimizer.pth``,
``critic.optimizer.pth``, ``pytorch_variables.pth``, ``_stable_baselines3_version``) and the real ``SACPolicy`` state-dict
layout, critics and target critics included -- SB3 itself is not installed here.  The ``data`` entry is JSON as SB3 writes
it: plain values as they are, objects as ``{":type:", ":serialized:"}`` cloudpickle records."""
import ctypes
import io
import json
import os
import re
import zipfile

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PICKLED = {":type:": "<class 'dict'>", ":serialized:": "gAWVKQAAAAAAAAB9lCiMCG5ldF9hcmNolF2UKEuAS4BlfZQu"}


@pytest.fixture(scope="module")
def mods():
    from fpv_drone_rl_agent_b200 import ppo, sac

    return ppo, sac


def _sac_state_dict(od=20, ad=4, h=(128, 128), seed=0, critic_h=256):
    """SACPolicy.state_dict() of SB3 2.x (MlpPolicy, share_features_extractor=False, n_critics=2)."""
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g) * 0.2  # noqa: E731
    sd = {"actor.latent_pi.0.weight": r(h[0], od), "actor.latent_pi.0.bias": r(h[0]),
          "actor.latent_pi.2.weight": r(h[1], h[0]), "actor.latent_pi.2.bias": r(h[1]),
          "actor.mu.weight": r(ad, h[1]) * 5, "actor.mu.bias": r(ad), "actor.log_std.weight": r(ad, h[1]), "actor.log_std.bias": r(ad)}
    for net in ("critic", "critic_target"):
        for q in ("qf0", "qf1"):
            sd.update({f"{net}.{q}.0.weight": r(critic_h, od + ad), f"{net}.{q}.0.bias": r(critic_h),
                       f"{net}.{q}.2.weight": r(critic_h, critic_h), f"{net}.{q}.2.bias": r(critic_h),
                       f"{net}.{q}.4.weight": r(1, critic_h), f"{net}.{q}.4.bias": r(1)})
    return sd


def _sac_data(policy_kwargs=None, use_sde=False):
    return {"policy_class": {":type:": "<class 'abc.ABCMeta'>", ":serialized:": "gAWVMAAAAAAAAACMHnN0YWJsZV9iYXNlbGluZXMzLnNhYy5wb2xpY2llc5Qu",
                             "__module__": "stable_baselines3.sac.policies"},
            "device": "auto", "verbose": 1, "policy_kwargs": {"net_arch": [128, 128], "use_sde": use_sde} if policy_kwargs is None else policy_kwargs,
            "num_timesteps": 200000, "_total_timesteps": 200000, "seed": None, "learning_rate": 0.0003, "buffer_size": 1000000,
            "batch_size": 256, "tau": 0.005, "gamma": 0.99, "ent_coef": "auto", "target_entropy": -4.0, "use_sde": use_sde,
            "observation_space": {":type:": "<class 'gymnasium.spaces.box.Box'>", ":serialized:": "gAWV", "dtype": "float64", "_shape": [20]},
            "action_space": {":type:": "<class 'gymnasium.spaces.box.Box'>", ":serialized:": "gAWV", "dtype": "float32", "_shape": [4]}}


def _torch_bytes(obj):
    buf = io.BytesIO()
    torch.save(obj, buf)
    return buf.getvalue()


def _write_archive(path, sd, data, optimizers=("actor.optimizer.pth", "critic.optimizer.pth")):
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("data", json.dumps(data))
        for name in optimizers:
            z.writestr(name, _torch_bytes({"state": {}, "param_groups": [{"lr": 3e-4, "params": [0, 1, 2]}]}))
        z.writestr("policy.pth", _torch_bytes(sd))
        z.writestr("pytorch_variables.pth", _torch_bytes({"log_ent_coef": torch.tensor([-1.5])}))
        z.writestr("_stable_baselines3_version", "2.7.0")
        z.writestr("system_info.txt", "- OS: Linux\n- Python: 3.12\n- Stable-Baselines3: 2.7.0\n")
    return str(path)


def _np_actor(sd, x):
    """SB3's deterministic actor restated in float64 numpy: tanh(mu(relu(W2 relu(W1 x + b1) + b2)))."""
    f = {k: v.double().numpy() for k, v in sd.items() if k.startswith("actor.")}
    h = np.maximum(x @ f["actor.latent_pi.0.weight"].T + f["actor.latent_pi.0.bias"], 0.0)
    h = np.maximum(h @ f["actor.latent_pi.2.weight"].T + f["actor.latent_pi.2.bias"], 0.0)
    return np.tanh(h @ f["actor.mu.weight"].T + f["actor.mu.bias"])


@pytest.mark.parametrize("od,ad,h", [(20, 4, (128, 128)), (12, 1, (64, 64)), (20, 4, (128, 64))])
def test_sac_archive_loads_the_actor(mods, tmp_path, od, ad, h):
    ppo, sac = mods
    sd = _sac_state_dict(od, ad, h)
    arc = sac.load_sb3_zip(_write_archive(tmp_path / "sac.zip", sd, _sac_data()))
    assert arc.algorithm == "SAC" and arc.sb3_version == "2.7.0" and arc.vecnormalize is None
    m = arc.model
    assert isinstance(m, sac.SacActor) and (m.obs_dim, m.act_dim, m.net_arch) == (od, ad, h)
    got = m.state_dict()
    assert set(got) == {k[len("actor."):] for k in sd if k.startswith("actor.")}
    for k, v in got.items():
        assert torch.equal(v, sd["actor." + k]), k
    # the torch forward against the float64 numpy restatement
    x = np.random.default_rng(1).normal(0, 2, (4096, od))
    ref = _np_actor(sd, x)
    with torch.no_grad():
        y64 = m.double()(torch.from_numpy(x)).numpy()
        y32 = m.float()(torch.from_numpy(x).float()).double().numpy()
    assert np.abs(y64 - ref).max() < 1e-12
    assert np.abs(y32 - ref).max() < 2e-5
    assert (np.abs(ref) > 0.5).mean() > 0.2, "the squash should be exercised"


def test_sac_activation_from_policy_kwargs(mods, tmp_path):
    """absent = ReLU (SAC's default); a named ReLU is accepted too"""
    _, sac = mods
    sd = _sac_state_dict()
    for kw in ({"net_arch": [128, 128]}, {"net_arch": [128, 128], "activation_fn": "torch.nn.ReLU"}, {}):
        assert sac.load_sb3_zip(_write_archive(tmp_path / "a.zip", sd, _sac_data(policy_kwargs=kw))).algorithm == "SAC"


@pytest.mark.parametrize("case,match", [
    ("pickled_kwargs", "policy_kwargs is stored as a cloudpickle"),
    ("tanh_sac", "SAC activation_fn 'torch.nn.Tanh' is not supported"),
    ("wide", "256 units wide; hidden widths above 128"),
    ("sde_data", "gSDE"),
    ("sde_kwargs", "gSDE"),
    ("sde_param", "gSDE log_std matrix"),
    ("three_layers", "has 3 linear layers"),
    ("wide_obs", "observation width 40 > 32"),
    ("wide_act", "action width 6 > 4"),
    ("no_policy", "no policy.pth"),
    ("unknown", "neither SAC actor keys"),
])
def test_sac_refusals(mods, tmp_path, case, match):
    _, sac = mods
    sd, data = _sac_state_dict(), _sac_data()
    if case == "pickled_kwargs":
        data["policy_kwargs"] = PICKLED
    elif case == "tanh_sac":
        data["policy_kwargs"] = {"net_arch": [128, 128], "activation_fn": "torch.nn.Tanh"}
    elif case == "wide":
        sd = _sac_state_dict(h=(256, 256))  # SB3's default SAC net_arch
    elif case == "sde_data":
        data = _sac_data(use_sde=True)
    elif case == "sde_kwargs":
        data["policy_kwargs"] = {"net_arch": [128, 128], "use_sde": True}
    elif case == "sde_param":
        sd = {k: v for k, v in sd.items() if not k.startswith("actor.log_std.")}
        sd["actor.log_std"] = torch.zeros(128, 4)
    elif case == "three_layers":
        sd["actor.latent_pi.4.weight"], sd["actor.latent_pi.4.bias"] = torch.zeros(128, 128), torch.zeros(128)
    elif case == "wide_obs":
        sd = _sac_state_dict(od=40)
    elif case == "wide_act":
        sd = _sac_state_dict(ad=6)
    elif case == "unknown":
        sd = {"q_net.0.weight": torch.zeros(4, 4)}
    path = tmp_path / f"{case}.zip"
    if case == "no_policy":
        with zipfile.ZipFile(path, "w") as z:
            z.writestr("data", json.dumps(data))
    else:
        _write_archive(path, sd, data)
    with pytest.raises(ValueError, match=re.escape(match)):
        sac.load_sb3_zip(str(path))


def _ppo_model(ppo, od, ad, hidden):
    torch.manual_seed(od + hidden)
    m = ppo.ActorCritic(od, ad, hidden=hidden, log_std_init=-0.4)
    with torch.no_grad():
        for lin in (m.pi1, m.pi2, m.vf1, m.vf2, m.mu, m.v):
            rows = hidden if lin.bias.numel() == ppo.HID else lin.bias.numel()
            lin.bias[:rows].uniform_(-0.3, 0.3)
    return m


@pytest.mark.parametrize("od,ad,hidden", [(20, 4, 128), (12, 1, 64)])
def test_ppo_export_import_round_trip(mods, tmp_path, od, ad, hidden):
    """export_sb3_zip -> load_sb3_zip gives the same ActorCritic bit for bit, and the VecNormalize arrays it carries"""
    ppo, sac = mods
    m = _ppo_model(ppo, od, ad, hidden)
    st, rt = ppo.RunningStats.__new__(ppo.RunningStats), ppo.RunningStats.__new__(ppo.RunningStats)
    g = torch.Generator().manual_seed(3)
    st.stats, st.dim, st.eps = torch.cat([torch.randn(od, generator=g, dtype=torch.float64), torch.rand(od, generator=g, dtype=torch.float64) + 0.1,
                                          torch.tensor([12345.0], dtype=torch.float64)]), od, 1e-8
    rt.stats, rt.dim, rt.eps = torch.tensor([0.0, 4.0, 99.0], dtype=torch.float64), 1, 1e-8
    vn = ppo.export_vecnormalize(st, rt, ppo.PPOConfig(clip_obs=7.0))
    path = str(tmp_path / "ppo.zip")
    ppo.export_sb3_zip(m, path, vn)
    arc = sac.load_sb3_zip(path)
    assert arc.algorithm == "PPO" and isinstance(arc.model, ppo.ActorCritic)
    assert (arc.model.obs_dim, arc.model.act_dim) == (od, ad)
    for k, v in m.state_dict().items():
        assert torch.equal(arc.model.state_dict()[k], v), k
    assert np.array_equal(arc.vecnormalize["obs_rms.mean"], vn["obs_rms"]["mean"])
    assert np.array_equal(arc.vecnormalize["obs_rms.var"], vn["obs_rms"]["var"])
    assert float(arc.vecnormalize["clip_obs"]) == 7.0 and bool(arc.vecnormalize["norm_obs"])
    # the same arrays through a separate .npz file (what tools/sb3_vecnormalize_to_npz.py writes)
    with zipfile.ZipFile(path) as z:
        (tmp_path / "vn.npz").write_bytes(z.read("vecnormalize.npz"))
    vn2 = sac.load_vecnormalize(str(tmp_path / "vn.npz"))
    assert set(vn2) == set(arc.vecnormalize) and all(np.array_equal(vn2[k], arc.vecnormalize[k]) for k in vn2)


@pytest.mark.parametrize("case,match", [
    ("relu", "PPO activation_fn 'torch.nn.ReLU' is not supported"),
    ("pickled_kwargs", "policy_kwargs is stored as a cloudpickle"),
    ("wide", "256 units wide"),
    ("sde", "gSDE"),
])
def test_ppo_refusals(mods, tmp_path, case, match):
    ppo, sac = mods
    m = _ppo_model(ppo, 20, 4, 128)
    sd = ppo.export_sb3_state_dict(m)
    data = {"policy_kwargs": {"net_arch": [128, 128]}, "use_sde": False}
    if case == "relu":
        data["policy_kwargs"]["activation_fn"] = "torch.nn.ReLU"
    elif case == "pickled_kwargs":
        data["policy_kwargs"] = PICKLED
    elif case == "wide":
        sd["mlp_extractor.policy_net.0.weight"] = torch.zeros(256, 20)
    elif case == "sde":
        sd["log_std"] = torch.zeros(128, 4)
    path = _write_archive(tmp_path / f"{case}.zip", sd, data, optimizers=("policy.optimizer.pth",))
    with pytest.raises(ValueError, match=re.escape(match)):
        sac.load_sb3_zip(path)


def test_sac_abi_and_argument_validation():
    """include/sac_b200.h's declarations are exported and bound; bad arguments come back as QX_EINVAL before anything
    touches CUDA (no GPU here)."""
    import __graft_entry__ as ge

    ge.build()
    from fpv_drone_rl_agent_b200 import _lib

    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "sac_b200.h")).read(), flags=re.S)
    names = sorted(set(re.findall(r"\b(sac_[a-z0-9_]+)\s*\(", src)))
    assert names == sorted(_lib.SAC_EXPORTED) == ["sac_actor_forward"]
    L = _lib.lib()
    good = dict(w1=0x10000, w2=0x20000, w_mu=0x30000, b1=0x40000, b2=0x50000, b_mu=0x60000, obs_dim=20, act_dim=4)
    obs, act = 0x70000, 0x80000

    def call(actor=None, obs_=obs, stride=20, n=256, mean=None, inv=None, actions=act, norm_out=None, **over):
        a = _lib.SacActor(**{**good, **over}) if actor is None else actor
        return L.sac_actor_forward(ctypes.byref(a), obs_, stride, n, mean, inv, 10.0, actions, norm_out, None)

    assert L.sac_actor_forward(None, obs, 20, 256, None, None, 10.0, act, None, None) == -1
    assert b"sac_actor_forward" in L.qx_last_error()
    for over in (dict(w1=0), dict(w2=0), dict(w_mu=0), dict(b1=0), dict(b2=0), dict(b_mu=0), dict(w1=0x10008), dict(w2=0x20004),
                 dict(w_mu=0x30002), dict(b1=0x40002), dict(obs_dim=0), dict(obs_dim=33), dict(act_dim=0), dict(act_dim=5)):
        assert call(**over) == -1, over
    for kw in (dict(obs_=None), dict(obs_=obs + 2), dict(n=0), dict(n=-1), dict(stride=19), dict(actions=None), dict(actions=act + 1),
               dict(norm_out=0x90001), dict(mean=0xA0000), dict(inv=0xB0000), dict(mean=0xA0002, inv=0xB0000)):
        assert call(**kw) == -1, kw


def test_sac_kernel_budget():
    """The SAC actor kernel keeps its four 128-thread slots without spilling (512 threads: at most 128 registers) and runs its
    layers on tcgen05.mma (UTCHMMA in the SASS)."""
    import importlib.util
    import subprocess

    import __graft_entry__ as ge

    ge.build()
    from fpv_drone_rl_agent_b200 import _lib

    csrc = os.path.dirname(_lib.LIB_PATH)
    log = os.path.join(csrc, "build.log")
    if not os.path.exists(log):  # library up to date but its log not in the checkout: rebuild once
        spec = importlib.util.spec_from_file_location("qx_build", os.path.join(csrc, "build.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.build(force=True)
    m = re.search(r"Compiling entry function '_ZN3sac20actor_forward_kernelENS_4ArgsE' for 'sm_100a'.*?(\d+) bytes spill stores, "
                  r"(\d+) bytes spill loads.*?Used (\d+) registers", open(log).read(), re.S)
    assert m and int(m.group(1)) == 0 and int(m.group(2)) == 0 and int(m.group(3)) <= 128, m and m.groups()
    lib = _lib.LIB_PATH
    try:
        sass = subprocess.run(["cuobjdump", "-sass", "-fun", "_ZN3sac20actor_forward_kernelENS_4ArgsE", lib], capture_output=True, text=True,
                              timeout=300).stdout
    except (FileNotFoundError, subprocess.TimeoutExpired):
        pytest.skip("cuobjdump not available")
    assert sass.count("UTCHMMA") >= 18 and "MUFU.TANH" not in sass
