"""GPU: the policy-forward kernel (ppo::policy_forward_kernel, K2) row by row against a float64 reference that rounds where
the kernel rounds, at training sizes, in the yaw shapes, in gather (time-limit bootstrap) mode and with the fused statistics.

The reference (``_Ref``) follows the kernel's rounding points in order:
  x_hat = clamp((x - mean) * inv_std, +-clip)           fp32, as the kernel computes it: obs_norm_out must equal it bit for bit
  X = bf16_rne(x_hat)
  p1 = fp32(fp32(X . W1^T in fp64) + b1);  h1 = hook(p1)  the kernel's own activation (ppo_test_tanh_bf16: bf16(tanh.approx))
  p2, h2 the same for layer 2
  [mean, value] = fp32(fp64 GEMM of h2 with W3) + b3
Products of bf16 values are exact in fp64, so what remains between kernel and reference is the tensor core's fp32
accumulation, which now and then moves a pre-activation across a bf16 rounding boundary of its activation (a one-ulp flip).
The acceptance rule (``_accept``) therefore has two parts: all but a small fraction of the rows agree to NEAR, and every row
lies within MAX, the effect of a few flips.  Both numbers were measured on a B200 (printed by the tests, see _TOL) and are
held with a 4x margin.  ``test_sensitivity`` shows that the rule fails, on many rows, for the mistakes it is there to catch.

The Gaussian noise is replayed with the oracle's Philox (key = seed ^ (row0 + row), counter (0, 3, step)) and the kernel's
Box-Muller; the only slack is the error bound of __logf / __sincosf / __expf.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

# name -> (obs_dim, act_dim, hidden)
SHAPES = {"hover128": (20, 4, 128), "hover64": (20, 4, 64), "yaw128": (12, 1, 128), "yaw64": (12, 1, 64)}
NEAR = 1e-5  # a row "agrees" when its action means and value are all within NEAR of the reference
# per shape: (largest fraction of rows allowed beyond NEAR, largest deviation of any row), 4x the largest a B200 (1000 W
# power limit) measured over every call of this file at 18 944 rows or more (the "measured" lines the tests print):
#   hover128 4.77e-3 / 2.92e-3,  hover64 1.04e-3 / 3.62e-3,  yaw128 3.77e-3 / 3.37e-3,  yaw64 9.0e-4 / 1.91e-3
# (exact tanh in place of tanh.approx, by comparison, puts 23-25 % of the rows beyond NEAR: test_sensitivity)
_TOL = {"hover128": (1.9e-2, 1.2e-2), "hover64": (4.2e-3, 1.45e-2), "yaw128": (1.5e-2, 1.35e-2), "yaw64": (3.6e-3, 7.6e-3)}
ROW_COUNTS = [1, 127, 128, 129, 18_944, 18_945, 56_832, 56_833, 131_072, 262_144 + 77, 1 << 20]
LOG_STD = [-0.5, 0.0, 0.3, -1.0]
TILE = 128


@pytest.fixture(scope="module")
def env():
    import __graft_entry__ as ge

    ge.build()
    from fpv_drone_rl_agent_b200 import _lib, ppo

    return _lib, ppo


def _model(ppo, shape, seed=0):
    """ActorCritic with non-trivial heads and biases (as test_gpu_ppo._model); the narrow embedding keeps its extra units zero."""
    od, ad, hid = SHAPES[shape]
    torch.manual_seed(seed)
    m = ppo.ActorCritic(od, ad, hidden=hid).cuda()
    with torch.no_grad():
        m.mu.weight.mul_(30.0)
        m.mu.bias.uniform_(-0.2, 0.2)
        m.v.bias.fill_(0.3)
        m.log_std.copy_(torch.tensor(LOG_STD[:ad]))
        for lin in (m.pi1, m.pi2, m.vf1, m.vf2):
            lin.bias[:hid].uniform_(-0.3, 0.3)
    return m


def _obs(n, od, stride, seed, scale=2.0):
    """[n, od] raw observations, a view of an [n, stride] buffer: spread wide enough that clip 3 bites."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    buf = torch.randn(n, stride, device="cuda", generator=g) * scale + torch.linspace(-1.5, 1.5, stride, device="cuda")
    return buf[:, :od]


def _norm(od, seed):
    g = torch.Generator(device="cuda").manual_seed(1000 + seed)
    return torch.randn(od, device="cuda", generator=g) * 0.3, torch.rand(od, device="cuda", generator=g) + 0.5


class _Ref:
    """float64 restatement of the kernel with its rounding points (module docstring); `mut` names a deliberate mistake."""

    def __init__(self, L, pol):
        self.L, self.pol = L, pol
        self.od, self.ad = pol.model.obs_dim, pol.model.act_dim
        self.w1, self.w2p, self.w2v, self.w3 = (w.double() for w in (pol.w1, pol.w2p, pol.w2v, pol.w3))
        self.b1, self.b2, self.b3 = pol.b1.clone(), pol.b2.clone(), pol.b3.clone()
        self.log_std = pol.log_std.double().clone()

    def hook(self, p):
        p = p.contiguous()
        out = torch.empty(p.shape, dtype=torch.int16, device=p.device)
        assert self.L.ppo_test_tanh_bf16(p.data_ptr(), out.data_ptr(), p.numel(), None) == 0
        return out.view(torch.bfloat16).double()

    def act(self, p, mut):
        if mut == "no_bf16":  # activations kept at full precision
            return torch.tanh(p.double())
        if mut == "exact_tanh":  # correctly rounded tanh in place of tanh.approx
            return torch.tanh(p.double()).to(torch.bfloat16).double()
        return self.hook(p)

    def normalize(self, obs, mean, inv_std, clip):
        x = obs.float()
        if mean is not None:
            x = (x - mean) * inv_std  # two fp32 roundings, as the kernel (no contraction)
        c = clip if clip > 0 else 3.0e38
        return x.clamp(-c, c)

    def forward(self, obs, mean=None, inv_std=None, clip=10.0, mut=None):
        """-> (x_hat fp32 [n, od], mean fp64 [n, ad], value fp64 [n])"""
        if mut == "neighbour_obs":
            obs = torch.roll(obs, 1, 0)
        elif mut == "tile_earlier":
            obs = torch.roll(obs, TILE, 0)
        xh = self.normalize(obs, mean, inv_std, clip)
        X = xh.to(torch.bfloat16).double()
        b1, b2 = self.b1.clone(), self.b2.clone()
        if mut == "drop_b1":  # the actor's first-layer unit with the largest bias loses it
            b1[int(b1[:128].abs().argmax())] = 0.0
        if mut == "drop_b2v":  # the critic's second-layer unit with the largest bias loses it
            b2[128 + int(b2[128:].abs().argmax())] = 0.0
        h1 = self.act((X @ self.w1[:, :self.od].t()).float() + b1, mut)
        h2p = self.act((h1[:, :128] @ self.w2p.t()).float() + b2[:128], mut)
        h2v = self.act((h1[:, 128:] @ self.w2v.t()).float() + b2[128:], mut)
        out = ((h2p @ self.w3[:, :128].t() + h2v @ self.w3[:, 128:].t()).float() + self.b3).double()
        vcol = {"value_col_plus": self.ad + 1, "value_col_minus": self.ad - 1}.get(mut, self.ad)
        return xh, out[:, :self.ad], out[:, vcol]


def _accept(dev, shape):
    """the acceptance rule for per-row deviations `dev` (max over the row's action means and value) -> (ok, n_far, max)"""
    frac, mx = _TOL[shape]
    n = dev.numel()
    n_far = int((dev > NEAR).sum())
    dmax = float(dev.max()) if n else 0.0
    return n_far <= frac * n + 3 and dmax <= mx, n_far, dmax


def _row_dev(mean_k, value_k, mean_r, value_r):
    return torch.maximum((mean_k.double() - mean_r).abs().amax(1), (value_k.double() - value_r).abs())


# ---------------------------------------------------------------------------------------------------------------------------
# noise replay
# ---------------------------------------------------------------------------------------------------------------------------
def _noise(n, seed, row0, step, trunc_gid=False, drop_step_hi=False):
    """the kernel's four standard-normal draws of rows 0..n-1 in float64 -> (z [n, 4], per-draw error bound [n, 4]);
    trunc_gid / drop_step_hi: the draws of a kernel that kept only 32 bits of row0 + row / of the step"""
    from oracle.quadx_model import philox4x32, u01

    with np.errstate(over="ignore"):
        gid = np.uint64(row0) + np.arange(n, dtype=np.uint64)
    if trunc_gid:
        gid = gid & np.uint64(0xFFFFFFFF)
    step_hi = 0 if drop_step_hi else (step >> 32) & 0xFFFFFFFF
    ctr = np.zeros((n, 4), np.uint32)
    ctr[:, 1], ctr[:, 2], ctr[:, 3] = 3, step & 0xFFFFFFFF, step_hi
    key = np.empty((n, 2), np.uint32)
    key[:, 0] = (np.uint64(seed & 0xFFFFFFFF) ^ (gid & np.uint64(0xFFFFFFFF))).astype(np.uint32)
    key[:, 1] = (np.uint64(seed >> 32) ^ (gid >> np.uint64(32))).astype(np.uint32)
    b = philox4x32(ctr, key, rounds=10)
    ua, ub = u01(b[:, 0]), u01(b[:, 2])
    # the angle exactly as the kernel forms it in fp32 (u01 is exact in fp32; no contraction)
    ang = [(np.float32(6.28318530718) * u01(b[:, k]).astype(np.float32) - np.float32(3.14159265359)).astype(np.float64) for k in (1, 3)]
    z = np.empty((n, 4))
    err = np.empty((n, 4))
    for j, (u, a) in enumerate(((ua, ang[0]), (ub, ang[1]))):
        Lg = -2.0 * np.log(u)
        rad = np.sqrt(Lg)
        # __logf: 2^-21.41 absolute on [0.5, 2], 3 ulp elsewhere; the approximate square root: a few fp32 ulp
        dL = 2.0 * (2.0 ** -21.41 + 3.0 * 2.0 ** -23 * np.abs(np.log(u)))
        drad = np.maximum(np.sqrt(Lg + dL) - rad, rad - np.sqrt(np.maximum(Lg - dL, 0.0))) + 2.0 ** -21 * rad
        z[:, 2 * j], z[:, 2 * j + 1] = -rad * np.cos(a), -rad * np.sin(a)
        e = drad + rad * 2.0 ** -21.41  # __sincosf: 2^-21.41 absolute on [-pi, pi]
        err[:, 2 * j] = err[:, 2 * j + 1] = e
    err += 2.0 ** -23 * np.abs(z)
    return z, err


def _check_noise(pol, z, zerr, act_s, env_s, logp_s, act_d, std_idx=None):
    """stochastic outputs against the replayed draws; act_d = the kernel's deterministic action means (checked separately
    against the reference).  Returns the number of rows that fail (0 = pass)."""
    ad = pol.model.act_dim
    ls = pol.log_std.double().cpu().numpy()
    idx = np.arange(ad) if std_idx is None else std_idx
    a_s, a_d = act_s.double().cpu().numpy(), act_d.double().cpu().numpy()
    std = np.exp(ls[idx])
    zj, ej = z[:, :ad], zerr[:, :ad]
    # a = fmaf(__expf(ls), nz, mean): the noise term std * z, then one fp32 rounding of the sum
    tol = std * (ej + 4.0 * 2.0 ** -23 * np.abs(zj)) + 2.0 ** -23 * (np.abs(a_s) + np.abs(a_d)) + 1e-7
    bad_a = (np.abs((a_s - a_d) - std * zj) > tol).any(1)
    lp_ref = (-0.5 * zj * zj - ls[idx] - 0.5 * math.log(2 * math.pi)).sum(1)
    lp_tol = (np.abs(zj) * ej).sum(1) + 1e-6 * (1.0 + np.abs(lp_ref) + (0.5 * zj * zj).sum(1))
    bad_lp = np.abs(logp_s.double().cpu().numpy() - lp_ref) > lp_tol
    assert torch.equal(env_s, act_s.clamp(-1.0, 1.0))
    return int((bad_a | bad_lp).sum())


# ---------------------------------------------------------------------------------------------------------------------------
def _outputs(n, od, ad):
    return dict(actions=torch.full((n, ad), 7.0, device="cuda"), env_actions=torch.full((n, ad), 7.0, device="cuda"),
                values=torch.full((n,), 7.0, device="cuda"), log_probs=torch.full((n,), 7.0, device="cuda"),
                obs_norm=torch.full((n, od), 7.0, device="cuda"))


def _run_and_check(ppo, ref, pol, obs, shape, *, mean=None, inv_std=None, clip=3.0, seed=5, row0=0, step=0, step_base=None,
                   base_add=0, label=""):
    """deterministic and stochastic call through ppo.policy_forward; every output of every row checked -> deviations"""
    od, ad, _ = SHAPES[shape]
    n = obs.shape[0]
    norm = (mean, inv_std) if mean is not None else None
    d, s = _outputs(n, od, ad), _outputs(n, od, ad)
    ppo.policy_forward(pol, obs, norm=norm, obs_clip=clip, deterministic=True, **d)
    ppo.policy_forward(pol, obs, norm=norm, obs_clip=clip, seed=seed, row0=row0, step=step, step_base=step_base, **s)
    xh, m_r, v_r = ref.forward(obs, mean, inv_std, clip)
    torch.cuda.synchronize()
    assert torch.equal(d["obs_norm"], xh) and torch.equal(s["obs_norm"], xh), "obs_norm_out is not the fp32 normalisation"
    assert torch.equal(d["env_actions"], d["actions"].clamp(-1.0, 1.0))
    assert torch.equal(s["values"], d["values"]), "values depend on the sampling"
    lp_det = float(-(ref.log_std[:ad].sum() + ad * 0.5 * math.log(2 * math.pi)))
    assert (d["log_probs"].double() - lp_det).abs().max().item() < 1e-5
    dev = _row_dev(d["actions"], d["values"], m_r, v_r)
    ok, n_far, dmax = _accept(dev, shape)
    print(f"measured {shape} {label} n={n}: rows beyond {NEAR:g}: {n_far} ({n_far / n:.2e}), max deviation {dmax:.3e}")
    assert ok, (shape, label, n, n_far, dmax)
    z, zerr = _noise(n, seed, row0, step + base_add)
    bad = _check_noise(pol, z, zerr, s["actions"], s["env_actions"], s["log_probs"], d["actions"])
    assert bad == 0, f"{bad} rows of {n} do not follow the Philox / Box-Muller draws"
    return d, s


def test_tanh_hook(env):
    """ppo_test_tanh_bf16 against float64 tanh: within one bf16 ulp of bf16_rne(tanh(x)) over a dense sweep of [-10, 10]
    (and the edges), low / high halves in place, and odd-symmetric bit for bit (as measured on a B200)."""
    _lib, ppo = env
    L = _lib.lib()
    g = torch.Generator(device="cuda").manual_seed(0)
    grid = torch.linspace(-10.0, 10.0, (1 << 24) + 1, device="cuda")
    bits = torch.randint(0, 1 << 31, (1 << 22,), device="cuda", generator=g, dtype=torch.int64).to(torch.int32).view(torch.float32)
    bits = bits[(bits <= 10.0) & (bits >= 1.1754944e-38)]  # every binade of (0, 10], down to the smallest normal (the kernel flushes subnormals)
    bits = torch.cat([bits, -bits])
    sat = torch.rand(1 << 20, device="cuda", generator=g) * 4.0 + 6.0
    edge = torch.tensor([0.0, -0.0, float("inf"), float("-inf"), 1e-30, -1e-30, 1e-8, -1e-8, 3e38, -3e38], device="cuda")
    x = torch.cat([grid, bits, sat, -sat, edge])
    x = x[torch.randperm(x.numel(), device="cuda", generator=g)]  # neighbours differ: a lo / hi swap could not hide
    x = torch.cat([x, torch.tensor([0.75], device="cuda")])  # odd length: the last element has no partner
    out = torch.empty(x.numel(), dtype=torch.int16, device="cuda")
    assert L.ppo_test_tanh_bf16(x.data_ptr(), out.data_ptr(), x.numel(), None) == 0
    torch.cuda.synchronize()
    h = out.view(torch.bfloat16).double()
    t = torch.tanh(x.double())
    r = t.to(torch.bfloat16).double()
    ulp = torch.where(r.abs() > 0, r.abs().log2().floor().exp2() * 2.0 ** -7, torch.full_like(r, 2.0 ** -133))
    miss = (h - r).abs()
    assert (miss <= ulp).all(), (x[miss > ulp][:8], h[miss > ulp][:8], r[miss > ulp][:8])
    assert torch.equal(h[x == float("inf")], torch.ones_like(h[x == float("inf")]))
    assert torch.equal(h[x == float("-inf")], -torch.ones_like(h[x == float("-inf")]))
    assert (h[x.abs() >= 9.0].abs() == 1.0).all()
    one_off = float((miss > 0).double().mean())
    mid = (x.abs() > 0.05) & (x.abs() < 3.0)  # where the hidden pre-activations live
    one_off_mid = float((miss[mid] > 0).double().mean())
    # odd symmetry
    xs = x[x.abs() > 0][: 1 << 22].contiguous()
    pos, neg = torch.empty(xs.numel(), dtype=torch.int16, device="cuda"), torch.empty(xs.numel(), dtype=torch.int16, device="cuda")
    xneg = (-xs).contiguous()
    assert L.ppo_test_tanh_bf16(xs.data_ptr(), pos.data_ptr(), xs.numel(), None) == 0
    assert L.ppo_test_tanh_bf16(xneg.data_ptr(), neg.data_ptr(), xs.numel(), None) == 0
    torch.cuda.synchronize()
    asym = (pos.view(torch.bfloat16).double() + neg.view(torch.bfloat16).double()) != 0
    print(f"measured tanh hook: one bf16 ulp from bf16_rne(tanh) for {one_off:.2e} of the sweep, {one_off_mid:.2e} of |x| in (0.05, 3); "
          f"{int(asym.sum())} of {xs.numel()} not odd-symmetric")
    assert int(asym.sum()) == 0  # measured on a B200: tanh.approx.f32 is odd-symmetric bit for bit


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("n", ROW_COUNTS)
def test_forward_matches_reference(env, shape, n):
    """Every row of every output: one tile, the first slot with two tiles (56 833 = 444 tiles + 1 row), training sizes.
    The row count also picks the input layout (stride obs_dim, 24 or obs_dim + 1) and the normalisation (statistics with
    clip 3, statistics with clip 0 = off, none)."""
    _lib, ppo = env
    od, ad, hid = SHAPES[shape]
    k = ROW_COUNTS.index(n)
    stride, mode = (od, 24, od + 1)[k % 3], (k // 3) % 3  # rows 1 .. 56 833 see all nine combinations
    m = _model(ppo, shape, seed=k)
    pol = ppo.PackedPolicy(m, "cuda")
    ref = _Ref(_lib.lib(), pol)
    obs = _obs(n, od, stride, seed=n)
    mean, inv = _norm(od, k)
    kw = [dict(mean=mean, inv_std=inv, clip=3.0), dict(mean=mean, inv_std=inv, clip=0.0), dict(mean=None, inv_std=None, clip=3.0)][mode]
    _run_and_check(ppo, ref, pol, obs, shape, seed=5 + k, row0=11 * k, step=3 + k, label=f"stride {stride} mode {mode}", **kw)


def test_counter_edges(env):
    """row0 + row crossing 2^32, step + *step_base crossing 2^32, a seed above 2^32: the replay holds, and the replay of a
    kernel that truncated the row id or the step to 32 bits would not."""
    _lib, ppo = env
    shape, n = "hover128", 128
    m = _model(ppo, shape)
    pol = ppo.PackedPolicy(m, "cuda")
    ref = _Ref(_lib.lib(), pol)
    obs = _obs(n, 20, 20, seed=3)
    mean, inv = _norm(20, 0)
    row0 = (1 << 32) - 64
    d, s = _run_and_check(ppo, ref, pol, obs, shape, mean=mean, inv_std=inv, seed=(1 << 40) + 12345, row0=row0, step=9, label="row0 2^32-64")
    z, e = _noise(n, (1 << 40) + 12345, row0, 9, trunc_gid=True)
    assert _check_noise(pol, z, e, s["actions"], s["env_actions"], s["log_probs"], d["actions"]) >= 60  # the 64 rows past 2^32
    base = torch.tensor([5], dtype=torch.int64, device="cuda")
    step = (1 << 32) - 2
    d, s = _run_and_check(ppo, ref, pol, obs, shape, mean=mean, inv_std=inv, seed=77, row0=0, step=step, step_base=base, base_add=5,
                          label="step 2^32+3")
    z, e = _noise(n, 77, 0, step + 5, drop_step_hi=True)
    assert _check_noise(pol, z, e, s["actions"], s["env_actions"], s["log_probs"], d["actions"]) >= n - 4


@pytest.mark.parametrize("shape", ["hover128", "yaw128"])
def test_sensitivity(env, shape):
    """The acceptance rule fails, on many rows, for each mistake it is there to catch (the kernel is not changed)."""
    _lib, ppo = env
    od, ad, _ = SHAPES[shape]
    n = 131_072
    m = _model(ppo, shape, seed=8)
    pol = ppo.PackedPolicy(m, "cuda")
    ref = _Ref(_lib.lib(), pol)
    obs = _obs(n, od, od, seed=8)
    mean, inv = _norm(od, 8)
    d, s = _run_and_check(ppo, ref, pol, obs, shape, mean=mean, inv_std=inv, clip=3.0, seed=1, row0=0, step=4, label="sensitivity")
    for mut in ("neighbour_obs", "tile_earlier", "drop_b1", "drop_b2v", "no_bf16", "exact_tanh", "value_col_plus", "value_col_minus"):
        _, m_r, v_r = ref.forward(obs, mean, inv, 3.0, mut=mut)
        ok, n_far, dmax = _accept(_row_dev(d["actions"], d["values"], m_r, v_r), shape)
        print(f"mutation {shape} {mut}: rows beyond {NEAR:g}: {n_far / n:.3f}, max deviation {dmax:.3e}")
        assert not ok and n_far >= n // 10, (mut, n_far, dmax)
    z, e = _noise(n, 1, 0, 4)
    shifted = (np.arange(ad) + 1) % 4
    assert _check_noise(pol, z, e, s["actions"], s["env_actions"], s["log_probs"], d["actions"], std_idx=shifted) >= n // 2
    swapped = np.arange(n) ^ 1  # the noise of neighbouring rows exchanged
    assert _check_noise(pol, z[swapped], e[swapped], s["actions"], s["env_actions"], s["log_probs"], d["actions"]) >= n // 2


def test_placement_invariance(env):
    """Deterministic outputs do not depend on where a row sits: the 1 Mi batch reversed, contiguous shards (row0 shifted: the
    stochastic actions follow the row id, not the position), and gather mode over a random permutation all give the full
    batch's rows bit for bit."""
    _lib, ppo = env
    L = _lib.lib()
    shape, n = "hover128", 1 << 20
    m = _model(ppo, shape, seed=4)
    pol = ppo.PackedPolicy(m, "cuda")
    obs = _obs(n, 20, 24, seed=4)
    st = ppo.RunningStats(20, "cuda")
    st.mean.copy_(_norm(20, 4)[0]); st.inv_std.copy_(_norm(20, 4)[1])

    def fwd(o, det=True, row0=0):
        out = _outputs(o.shape[0], 20, 4)
        ppo.policy_forward(pol, o, obs_stats=st, obs_clip=3.0, deterministic=det, seed=9, row0=row0, step=2, **out)
        return out

    full, full_s = fwd(obs), fwd(obs, det=False)
    rev = fwd(obs.flip(0).contiguous())
    torch.cuda.synchronize()
    for k in ("actions", "values", "obs_norm"):
        assert torch.equal(rev[k].flip(0), full[k]), k
    for a, b in ((0, 1000), (1000, 18_945), (18_945, 400_001), (400_001, n)):
        sh, sh_s = fwd(obs[a:b]), fwd(obs[a:b], det=False, row0=a)
        torch.cuda.synchronize()
        for k in ("actions", "values", "obs_norm"):
            assert torch.equal(sh[k], full[k][a:b]), (a, b, k)
        assert torch.equal(sh_s["actions"], full_s["actions"][a:b]) and torch.equal(sh_s["log_probs"], full_s["log_probs"][a:b])
    # gather mode: every row listed once, in random order; with gamma = 1 the stored gamma * V is V itself
    perm = torch.randperm(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4)).to(torch.int32)
    cnt = torch.tensor([n], dtype=torch.int32, device="cuda")
    te, tr = torch.zeros(n, dtype=torch.uint8, device="cuda"), torch.ones(n, dtype=torch.uint8, device="cuda")
    out = torch.full((n,), 7.0, device="cuda")
    assert L.ppo_bootstrap_truncated_first(C.byref(pol.struct), obs.data_ptr(), obs.stride(0), n, st.mean.data_ptr(), st.inv_std.data_ptr(), 3.0,
                                           cnt.data_ptr(), perm.data_ptr(), te.data_ptr(), tr.data_ptr(), 1.0, out.data_ptr(), None) == 0
    torch.cuda.synchronize()
    assert torch.equal(out, full["values"])


def _fma_f32(a, b, c):
    """fp32 fmaf(a, b, c) for fp32 arrays, rounded once: the product is exact in fp64; the fp64 sum is corrected where its
    own rounding could decide the fp32 tie"""
    a, b, c = (np.asarray(t, np.float64) for t in (a, b, c))
    p = a * b
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)  # TwoSum: s + err == p + c exactly
    r = s.astype(np.float32)
    lo = np.nextafter(r, np.float32(-np.inf)).astype(np.float64)
    hi = np.nextafter(r, np.float32(np.inf)).astype(np.float64)
    tie = ((s - r.astype(np.float64)) * 2 == (hi - r)) | ((s - r.astype(np.float64)) * 2 == (lo - r))
    fix = tie & (err != 0)
    s[fix] = np.nextafter(s[fix], np.where(err[fix] > 0, np.inf, -np.inf))
    return s.astype(np.float32)


@pytest.mark.parametrize("first", [False, True])
@pytest.mark.parametrize("shape", ["hover128", "yaw128"])
def test_bootstrap_gather(env, shape, first):
    """ppo_bootstrap_truncated(_first) over synthetic done queues in random order at n = 131 072: the listed rows that were
    truncated and not terminated get fmaf(gamma, V, r) (gamma V for _first) with V the forward's value of that row (itself
    checked against the reference); every other reward is untouched, also where truncated is set but the row is not listed."""
    _lib, ppo = env
    L = _lib.lib()
    od, ad, _ = SHAPES[shape]
    n, gamma = 131_072, 0.99
    m = _model(ppo, shape, seed=6)
    pol = ppo.PackedPolicy(m, "cuda")
    ref = _Ref(L, pol)
    obs = _obs(n, od, od + 1, seed=6)
    mean, inv = _norm(od, 6)
    d, _ = _run_and_check(ppo, ref, pol, obs, shape, mean=mean, inv_std=inv, clip=3.0, label="bootstrap")
    V = d["values"].cpu().numpy()
    g = torch.Generator(device="cuda").manual_seed(7)
    for count in (0, 1, 127, 128, 129, 18_945, 56_833, n):
        idx = torch.randperm(n, device="cuda", generator=g)[:count].to(torch.int32)
        idx_buf = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        idx_buf[:count] = idx
        cnt = torch.tensor([count], dtype=torch.int32, device="cuda")
        te = (torch.rand(n, device="cuda", generator=g) < 0.3).to(torch.uint8)
        tr = (torch.rand(n, device="cuda", generator=g) < 0.7).to(torch.uint8)
        r0 = torch.randn(n, device="cuda", generator=g)
        rew = r0.clone()
        fn = L.ppo_bootstrap_truncated_first if first else L.ppo_bootstrap_truncated
        assert fn(C.byref(pol.struct), obs.data_ptr(), obs.stride(0), n, mean.data_ptr(), inv.data_ptr(), 3.0, cnt.data_ptr(), idx_buf.data_ptr(),
                  te.data_ptr(), tr.data_ptr(), gamma, rew.data_ptr(), None) == 0
        torch.cuda.synchronize()
        listed = torch.zeros(n, dtype=torch.bool, device="cuda")
        listed[idx.long()] = True
        hit = (listed & tr.bool() & ~te.bool()).cpu().numpy()
        got, r0n = rew.cpu().numpy(), r0.cpu().numpy()
        assert np.array_equal(got[~hit].view(np.uint32), r0n[~hit].view(np.uint32)), count
        if first:
            exp = (np.float64(np.float32(gamma)) * V[hit]).astype(np.float32)
        else:
            exp = _fma_f32(np.full(int(hit.sum()), np.float32(gamma)), V[hit], r0n[hit])
        assert np.array_equal(got[hit].view(np.uint32), exp.view(np.uint32)), (count, int((got[hit] != exp).sum()))
        if 127 <= count < n:  # the queue is what counts: truncated rows that are not listed stay untouched
            assert (tr.bool() & ~te.bool() & ~listed).any() and hit.any()


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("shape", ["hover128", "yaw128"])
@pytest.mark.parametrize("n", [131_072, 262_144 + 77, 1 << 20])
def test_forward_stats(env, shape, fused, n):
    """ppo_policy_forward_stats (fused: merge inside the policy launch; chained: statistics launch + programmatic dependent),
    three successive batches: fp64 {mean, var, count} as a numpy VecNormalize merge, the fp32 (mean, inv_std) the exact casts
    of the kernel's fp64 statistics, the outputs row by row against the reference with those fp32 values, and the ticket /
    flag words re-armed after every call."""
    _lib, ppo = env
    od, ad, _ = SHAPES[shape]
    L = _lib.lib()
    m = _model(ppo, shape, seed=2)
    pol = ppo.PackedPolicy(m, "cuda")
    ref = _Ref(L, pol)
    st = ppo.RunningStats(od, "cuda")
    mu, var, count = np.zeros(od), np.ones(od), 1e-4
    eps = float(np.float32(st.eps))
    words = 148 * 64 * 2  # int32 index of the ticket word (ppo_running_stats_scratch_bytes: 148 x 64 partial sums, then the words)
    for rep in range(3):
        x = _obs(n, od, 24, seed=n + rep, scale=1.0 + rep)
        out = _outputs(n, od, ad)
        ppo.policy_forward(pol, x, obs_stats=st, obs_clip=5.0, seed=3, row0=rep * n, step=rep, update_stats=True, fused_stats=fused, **out)
        torch.cuda.synchronize()
        xd = x.double().cpu().numpy()
        bm, bv, bc = xd.mean(0), xd.var(0), n  # VecNormalize RunningMeanStd.update
        delta, tot = bm - mu, count + bc
        m2 = var * count + bv * bc + delta ** 2 * count * bc / tot
        mu, var, count = mu + delta * bc / tot, m2 / tot, tot
        s = st.stats.cpu().numpy()
        np.testing.assert_allclose(s[:od], mu, rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(s[od:2 * od], var, rtol=1e-7)
        assert abs(s[2 * od] - count) < 1e-6 * count
        assert torch.equal(st.mean, st.stats[:od].float())
        assert torch.equal(st.inv_std, (1.0 / torch.sqrt(st.stats[od:2 * od] + eps)).float())
        assert st.scratch.view(torch.int32)[words:words + 6].abs().sum().item() == 0, "ticket / flag words not re-armed"
        xh, m_r, v_r = ref.forward(x, st.mean, st.inv_std, 5.0)
        assert torch.equal(out["obs_norm"], xh)
        d = _outputs(n, od, ad)
        ppo.policy_forward(pol, x, norm=(st.mean, st.inv_std), obs_clip=5.0, deterministic=True, **d)
        torch.cuda.synchronize()
        assert torch.equal(d["values"], out["values"])
        dev = _row_dev(d["actions"], d["values"], m_r, v_r)
        ok, n_far, dmax = _accept(dev, shape)
        print(f"measured {shape} stats fused={fused} n={n} call {rep}: rows beyond {NEAR:g}: {n_far / n:.2e}, max deviation {dmax:.3e}")
        assert ok, (n_far, dmax)
        z, e = _noise(n, 3, rep * n, rep)
        assert _check_noise(pol, z, e, out["actions"], out["env_actions"], out["log_probs"], d["actions"]) == 0


@pytest.mark.parametrize("shape", ["hover128", "yaw128"])
def test_misaligned_buffers_take_the_scalar_paths(env, shape):
    """A column slice of a wider buffer (base + 1 float, stride 24) and outputs at a storage offset of one float give the
    aligned results bit for bit (the vector loads / stores need a 16-byte-aligned base, and fall back to scalar ones)."""
    _lib, ppo = env
    od, ad, _ = SHAPES[shape]
    n = 56_833
    pol = ppo.PackedPolicy(_model(ppo, shape, seed=5), "cuda")
    mean, inv = _norm(od, 5)
    aligned = _obs(n, od, 24, seed=5)
    buf = torch.zeros(n, 24, device="cuda")
    buf[:, 1:1 + od] = aligned
    shifted = buf[:, 1:1 + od]
    assert shifted.data_ptr() % 16 == 4 and shifted.stride(0) == 24

    def odd(shape_):  # contiguous, storage offset of one float
        numel = int(np.prod(shape_))
        return torch.full((numel + 1,), 7.0, device="cuda")[1:].view(shape_)

    for det in (True, False):
        base = _outputs(n, od, ad)
        ppo.policy_forward(pol, aligned, norm=(mean, inv), obs_clip=3.0, deterministic=det, seed=2, step=1, **base)
        for o, outs in ((shifted, _outputs(n, od, ad)), (aligned, None), (shifted, None)):
            outs = outs or dict(actions=odd((n, ad)), env_actions=odd((n, ad)), values=odd((n,)), log_probs=odd((n,)), obs_norm=odd((n, od)))
            ppo.policy_forward(pol, o, norm=(mean, inv), obs_clip=3.0, deterministic=det, seed=2, step=1, **outs)
            torch.cuda.synchronize()
            for k in base:
                assert torch.equal(outs[k], base[k]), (det, k)


def test_policy_forward_rejects_bad_outputs(env):
    """ppo.policy_forward refuses an output the kernel would write wrongly: not contiguous, wrong size, dtype or device."""
    _lib, ppo = env
    n = 256
    pol = ppo.PackedPolicy(_model(ppo, "hover128"), "cuda")
    obs = _obs(n, 20, 20, seed=1)
    bad = {
        "obs_norm": [torch.zeros(n, 24, device="cuda")[:, :20], torch.zeros(n, 21, device="cuda"), torch.zeros(n, 20, device="cuda", dtype=torch.float64)],
        "actions": [torch.zeros(n, 8, device="cuda")[:, :4], torch.zeros(n, 3, device="cuda"), torch.zeros(n, 4)],
        "env_actions": [torch.zeros(4, n, device="cuda").t(), torch.zeros(n + 1, 4, device="cuda")],
        "values": [torch.zeros(2 * n, device="cuda")[::2], torch.zeros(n - 1, device="cuda"), torch.zeros(n, device="cuda", dtype=torch.bfloat16)],
        "log_probs": [torch.zeros(n, 2, device="cuda")[:, 0], torch.zeros(n, 4, device="cuda")],
    }
    for name, ts in bad.items():
        for t in ts:
            with pytest.raises(ValueError, match=name):
                ppo.policy_forward(pol, obs, **{name: t})
    ok = torch.zeros(n, 4, device="cuda")  # [n * act_dim] flat is the same memory: accepted
    ppo.policy_forward(pol, obs, deterministic=True, actions=ok, values=torch.zeros(n, 1, device="cuda"))
    torch.cuda.synchronize()
