"""GPU: size-independent properties of the env-step path at BASELINE.json's
full sizes (1 Mi envs), where the float64 oracle is too slow to follow."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
HOVER_THR = float(np.sqrt(0.1 * 9.81 / 4.0))


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge

    ge.build()
    import fpv_drone_rl_agent_b200 as pkg

    return pkg


def _cfg(pkg, **kw):
    cfg = pkg.default_config()
    cfg.update(start_pos=[0, 0, 1.0], spawn_throttle=HOVER_THR, reset_idle_steps=0, **kw)
    return cfg


def _run(pkg, n, steps, seed, env_id0=0, k_fused=1, actions=None, bf16=False):
    sim = pkg.QuadXSim(n, _cfg(pkg), seed=seed, env_id0=env_id0)
    d = sim.device
    obs = torch.zeros(n, 20, device=d, dtype=torch.bfloat16 if bf16 else torch.float32)
    rew = torch.zeros(steps, n, device=d)
    te = torch.zeros(steps, n, dtype=torch.uint8, device=d)
    tr = torch.zeros(steps, n, dtype=torch.uint8, device=d)
    sim.reset(obs)
    if k_fused == 1:
        for k in range(steps):
            sim.step(actions[k], obs, rew[k], te[k], tr[k])
        last = obs.float()
    else:
        allobs = torch.zeros(steps, n, 20, device=d)
        for k in range(0, steps, k_fused):
            sim.step_k(actions[k:k + k_fused], allobs[k:k + k_fused], rew[k:k + k_fused], te[k:k + k_fused], tr[k:k + k_fused])
        last = allobs[-1]
    torch.cuda.synchronize()
    st = sim.get_state()
    sim.close()
    return last.cpu().numpy(), rew.cpu().numpy(), te.cpu().numpy(), tr.cpu().numpy(), st


def _actions(n, steps, device, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    a = torch.rand(steps, n, 4, generator=g) * 2 - 1
    a[..., :3] *= 0.3
    a[..., 3] = (2 * HOVER_THR - 1) + 0.3 * a[..., 3]  # SURVEY 8d C2: thrust centred on hover
    return a.to(device).contiguous()


def test_full_size_determinism_and_sharding(pkg):
    """1 Mi envs: (1) two runs are bit-identical; (2) splitting the env range over
    4 shards with env_id0 offsets gives bit-identical results (the Philox key is
    the global env id), which is what the multi-GPU path relies on."""
    n, steps = 1 << 20, 6
    a = _actions(n, steps, "cuda")
    o1, r1, te1, tr1, s1 = _run(pkg, n, steps, seed=77, actions=a)
    o2, r2, te2, tr2, s2 = _run(pkg, n, steps, seed=77, actions=a)
    assert np.array_equal(o1, o2) and np.array_equal(r1, r2) and np.array_equal(te1, te2)
    for k in s1:
        assert np.array_equal(s1[k], s2[k]), k
    q = n // 4
    for sh in range(4):
        o, r, te, tr, s = _run(pkg, q, steps, seed=77, env_id0=sh * q, actions=a[:, sh * q:(sh + 1) * q].contiguous())
        assert np.array_equal(o, o1[sh * q:(sh + 1) * q]) and np.array_equal(r, r1[:, sh * q:(sh + 1) * q])
    # different seeds / env ids really give different noise
    o3, r3, *_ = _run(pkg, 4096, steps, seed=78, actions=a[:, :4096].contiguous())
    assert not np.array_equal(r3, r1[:, :4096])
    assert np.isfinite(o1).all() and np.isfinite(r1).all()
    nq = np.sqrt(s1["qx"] ** 2 + s1["qy"] ** 2 + s1["qz"] ** 2 + s1["qw"] ** 2)
    assert np.abs(nq - 1).max() < 1e-5  # quaternion renormalisation


def test_step_k_equals_k_steps(pkg):
    """qx_step_k (k steps per launch, inline reset) against k x qx_step (deferred reset): two different kernel
    instantiations of the same arithmetic.  Flags must be identical; floats agree to fp32 rounding except where a
    camera pixel count flips (hover.py:209-213: the bbox ratio is a quotient of pixel counts, so a corner within
    rounding of a pixel boundary moves ratio / visibility / reward) -- allowed for < 0.1 % of the samples."""
    n, steps = 8192, 24
    a = _actions(n, steps, "cuda", seed=3)
    o1, r1, te1, tr1, s1 = _run(pkg, n, steps, seed=5, actions=a)
    o2, r2, te2, tr2, s2 = _run(pkg, n, steps, seed=5, actions=a, k_fused=8)
    assert np.array_equal(te1, te2) and np.array_equal(tr1, tr2)

    def close(x, y, tol, what):
        d = np.abs(x.astype(np.float64) - y.astype(np.float64))
        frac = float((d > tol).mean())
        assert frac < 1e-3, f"{what}: {frac:.2e} of the elements differ by more than {tol}"

    close(r1, r2, 1e-4, "reward")
    close(o1[:, 3:], o2[:, 3:], 2e-4, "obs")
    close(o1[:, :3], o2[:, :3], 5e-3, "obs ang_vel (Euler finite difference / 0.025, hover.py:228-230)")
    for k in s1:
        if s1[k].dtype.kind == "f":
            close(s1[k], s2[k], 1e-4, k)
        else:
            assert np.array_equal(s1[k], s2[k]), k


def test_bf16_obs_is_rounded_f32_obs(pkg):
    n, steps = 4096, 5
    a = _actions(n, steps, "cuda", seed=4)
    o1, r1, *_ = _run(pkg, n, steps, seed=6, actions=a)
    o2, r2, *_ = _run(pkg, n, steps, seed=6, actions=a, bf16=True)
    assert np.array_equal(r1, r2)
    assert np.array_equal(torch.from_numpy(o1).to(torch.bfloat16).float().numpy(), o2)


def test_episode_accounting_at_scale(pkg):
    """Zero thrust from the floor: every env ends on its 32nd step; the Monitor
    sums must say so exactly (a checksum over 256 Ki episodes)."""
    n = 1 << 18
    env = pkg.QuadXHoverVecEnv(n, seed=2, infos=False)
    env.reset()
    a = torch.zeros(n, 4, device=env.device)
    a[:, 3] = -1
    done_at = []
    for k in range(34):
        _, _, d, _ = env.step(a)
        c = int(d.sum())
        if c:
            assert c == n
            done_at.append(k)
    s, l, c = env.episode_stats()
    assert done_at == [31] and c == n and l == 32 * n
    assert -101.5 * n < s - (-30.0 * n) < -50.0 * n  # 31 shaped steps + one -100
    env.close()


def test_chunked_host_pipeline_equals_device_path(pkg):
    """qx_step_host cuts batches >= 2^17 into 8 chunks pipelined over three streams (H2D | kernels | D2H); the results
    must be those of the plain device-buffer call, including across a mass termination (reset queue per chunk), with
    pinned and with pageable host buffers, for a batch size that is not a multiple of anything.  qx_step_host_ex with
    bf16 observations (the compact wire format) must return the f32 observations rounded to nearest-even."""
    n = (1 << 17) + 37
    cfg = pkg.default_config()
    sim_h = pkg.QuadXSim(n, cfg, seed=3)
    sim_d = pkg.QuadXSim(n, pkg.default_config(), seed=3)
    d = sim_d.device
    obs = torch.zeros(n, 20, device=d); rew = torch.zeros(n, device=d)
    te = torch.zeros(n, dtype=torch.uint8, device=d); tr = torch.zeros_like(te)
    sim_d.reset(obs)
    torch.cuda.synchronize()
    assert np.array_equal(sim_h.reset_host(), obs.cpu().numpy())
    import ctypes as C

    from fpv_drone_rl_agent_b200 import _lib

    L = _lib.lib()
    a_pin = torch.zeros(n, 4).pin_memory(); o_pin = torch.zeros(n, 20).pin_memory(); r_pin = torch.zeros(n).pin_memory()
    te_pin = torch.zeros(n, dtype=torch.uint8).pin_memory(); tr_pin = torch.zeros(n, dtype=torch.uint8).pin_memory()
    o16_pin = torch.zeros(n, 20, dtype=torch.bfloat16).pin_memory()
    g = torch.Generator().manual_seed(0)
    for k in range(34):  # zero thrust: every env terminates on its 32nd step
        a = torch.rand(n, 4, generator=g) * 0.2 - 0.1
        a[:, 3] = -1.0
        sim_d.step(a.to(d), obs, rew, te, tr)
        torch.cuda.synchronize()
        if k % 3 == 2:  # compact wire format: bf16 observations, pinned buffers
            a_pin.copy_(a)
            _lib.check(L.qx_step_host_ex(sim_h._h, C.c_void_p(a_pin.data_ptr()), C.c_void_p(o16_pin.data_ptr()), 1, C.c_void_p(r_pin.data_ptr()),
                                         C.c_void_p(te_pin.data_ptr()), C.c_void_p(tr_pin.data_ptr()), None))
            assert torch.equal(obs.cpu().to(torch.bfloat16), o16_pin), k
            assert np.array_equal(rew.cpu().numpy(), r_pin.numpy()), k
            assert np.array_equal(te.cpu().numpy(), te_pin.numpy()) and np.array_equal(tr.cpu().numpy(), tr_pin.numpy()), k
            if k == 31:
                assert te_pin.numpy().all()
            continue
        if k % 3 == 0:  # pinned buffers, used in place
            a_pin.copy_(a)
            _lib.check(L.qx_step_host(sim_h._h, C.c_void_p(a_pin.data_ptr()), C.c_void_p(o_pin.data_ptr()), C.c_void_p(r_pin.data_ptr()),
                                      C.c_void_p(te_pin.data_ptr()), C.c_void_p(tr_pin.data_ptr()), None))
            o2, r2, te2, tr2 = o_pin.numpy(), r_pin.numpy(), te_pin.numpy().astype(bool), tr_pin.numpy().astype(bool)
        else:  # pageable numpy buffers through the staging area
            o2, r2, te2, tr2, _ = sim_h.step_host(a.numpy())
        assert np.array_equal(obs.cpu().numpy(), o2) and np.array_equal(rew.cpu().numpy(), r2), k
        assert np.array_equal(te.cpu().numpy().astype(bool), te2) and np.array_equal(tr.cpu().numpy().astype(bool), tr2), k
        if k == 31:
            assert te2.all()
    assert L.qx_step_host_ex(sim_h._h, C.c_void_p(a_pin.data_ptr()), C.c_void_p(o16_pin.data_ptr()), 7, None, None, None, None) != 0  # unknown dtype
    sa, sb = sim_h.get_state(), sim_d.get_state()
    for key in sa:
        assert np.array_equal(sa[key], sb[key]), key
    assert sim_h.episode_stats()[1:] == sim_d.episode_stats()[1:] == (32 * n, n)


def test_reference_constant_kernels_equal_generic_kernels(pkg, monkeypatch):
    """The kernels specialised for the reference's own parameter set (model constants as literals, qx_ref_constants.cuh)
    against the generic kernels that read every constant from the config: same config, same seeds, same actions.  The
    arithmetic is the same IEEE operations on the same values; only constant folding (x * 1, x * -1, fused constants) may
    differ, so the bound is a few ulp of the observation scale, and the flags are identical."""
    n, steps = 1 << 16, 96
    cfg = pkg.default_config()  # floor start, 10 idle steps per reset, auto-reset: every kernel mode runs
    g = torch.Generator(device="cuda").manual_seed(7)
    acts = (torch.rand(steps, n, 4, device="cuda", generator=g) * 2 - 1) * torch.tensor([0.3, 0.3, 0.3, 1.0], device="cuda")
    acts[..., 3] = acts[..., 3] * 0.3 + 0.1
    out = []
    for generic in (False, True):
        if generic:
            monkeypatch.setenv("QX_FORCE_GENERIC", "1")
        sim = pkg.QuadXSim(n, cfg, seed=99)
        assert sim.lib.qx_uses_reference_constants(sim._h) == (0 if generic else 1)
        d = sim.device
        obs = torch.zeros(n, 20, device=d); rew = torch.zeros(steps, n, device=d)
        te = torch.zeros(steps, n, dtype=torch.uint8, device=d); tr = torch.zeros(steps, n, dtype=torch.uint8, device=d)
        allobs = torch.zeros(steps, n, 20, device=d)
        sim.reset(obs)
        for k in range(steps):
            sim.step(acts[k], allobs[k], rew[k], te[k], tr[k])
        torch.cuda.synchronize()
        out.append((allobs.clone(), rew.clone(), te.clone(), tr.clone(), sim.episode_stats()))
        sim.close()
    (o1, r1, te1, tr1, s1), (o2, r2, te2, tr2, s2) = out
    assert torch.equal(te1, te2) and torch.equal(tr1, tr2) and s1[1:] == s2[1:]
    assert int(te1.sum()) > n  # episodes ended and restarted along the way
    # a few-ulp difference can move a projected panel edge across a pixel boundary (hover.py:209-213 counts pixels): those
    # samples differ by one pixel's worth in the camera features and the reward; they are counted, everything else is tight
    cam = [7, 8, 9, 10, 11, 12, 13, 14, 15]
    rest = [c for c in range(20) if c not in cam]
    flip = ((o1[..., cam] - o2[..., cam]).abs() > 1e-4).any(-1)
    n_flip, total = int(flip.sum()), flip.numel()
    do = float((o1[..., rest] - o2[..., rest]).abs().max())
    dcam = float((o1[..., cam] - o2[..., cam]).abs()[~flip].max())
    dr = float((r1 - r2).abs()[~flip].max())
    print(f"specialised vs generic kernels: max |obs diff| {do:.3e} (camera columns {dcam:.3e}), max |reward diff| {dr:.3e}, "
          f"pixel-count flips {n_flip}/{total}, bitwise equal: {torch.equal(o1, o2) and torch.equal(r1, r2)}")
    assert do <= 1e-4 and dr <= 1e-3 and n_flip <= 1e-4 * total
    assert float((o1 - o2).abs().max()) <= 0.2 and float((r1 - r2).abs().max()) <= 0.5  # a flip is one pixel row / column, not more


def test_inline_reset_equals_reset_queue_path(pkg):
    """qx_step resets finished envs inside the step launch for small batches (<= 16 384 envs) and through the deferred
    reset queue (qx_step_begin + qx_step_end, what the PPO rollout always uses) otherwise: same flags, same episode
    accounting, observations / rewards equal up to the rounding of two instantiations, through two mass terminations."""
    n, steps = 4096, 70
    cfg = pkg.default_config()  # floor start: every env is terminated by the floor rule on its 32nd step
    a = torch.tensor([[0.0, 0.0, 0.0, -1.0]], device="cuda").repeat(n, 1)
    outs = []
    for split in (False, True):
        sim = pkg.QuadXSim(n, cfg, seed=17)
        d = sim.device
        obs = torch.zeros(steps, n, 20, device=d); tobs = torch.zeros(steps, n, 20, device=d)
        rew = torch.zeros(steps, n, device=d)
        te = torch.zeros(steps, n, dtype=torch.uint8, device=d); tr = torch.zeros(steps, n, dtype=torch.uint8, device=d)
        o0 = torch.zeros(n, 20, device=d)
        sim.reset(o0)
        for k in range(steps):
            sim.step(a, obs[k], rew[k], te[k], tr[k], tobs[k], split=split)
        torch.cuda.synchronize()
        outs.append((obs, rew, te, tr, tobs, sim.episode_stats()))
        sim.close()
    (o1, r1, te1, tr1, t1, s1), (o2, r2, te2, tr2, t2, s2) = outs
    assert torch.equal(te1, te2) and torch.equal(tr1, tr2) and int(te1.sum()) == 2 * n
    assert s1[1:] == s2[1:] and abs(s1[0] - s2[0]) <= 1e-4 * abs(s2[0])
    assert float((o1 - o2).abs().max()) <= 1e-4 and float((r1 - r2).abs().max()) <= 1e-3
    done = te1.bool()
    assert float((t1[done] - t2[done]).abs().max()) <= 1e-4  # terminal observations of the finished envs


def test_step_kernel_variants_are_bitwise_equal(pkg, monkeypatch):
    """The sub-step code exists for three lane types: float = one env per thread on scalar instructions (csrc/qx_lanes.cuh),
    float2 = two envs per thread on packed FFMA2 / FMUL2 / FADD2, and S1 = one env per thread with its own components
    paired on the same packed instructions (csrc/qx_model.cuh, CoreS).  They are instantiated in the generic step kernel
    (any k, inline or queued reset), in the lean one-step kernel with a separate reset-queue launch, and in the merged
    launch (the last resident wave of blocks drains the reset queue); queued envs are re-created by the paired code or the
    generic one (QX_PAIRED_RESET), in one of four launch shapes (QX_SHAPE), with or without programmatic dependent launches
    (QX_PDL) and evict-first stores (QX_STREAM_STORES).  All perform the same IEEE operations per env, so they must agree
    bit for bit -- states, observations, terminal observations, rewards, flags, episode statistics -- through resets, for a
    batch size that leaves a thread with a single env, with the reference constants and with the generic constants.  The
    done queue of every step is exact on every variant.  bf16 observations written into a stride-32 policy buffer through
    the resets are the f32 ones rounded, on both reset paths."""
    from tests.util import check_done_queue

    n, steps = 40000 + 77, 70
    g = torch.Generator(device="cuda").manual_seed(11)
    acts = (torch.rand(steps, n, 4, device="cuda", generator=g) * 2 - 1) * torch.tensor([0.5, 0.5, 0.5, 1.0], device="cuda")
    acts[..., 3] = acts[..., 3] * 0.4 + 0.05
    paired4 = {"QX_HOT": "1", "QX_LANES": "4", "QX_MERGED": "0"}
    variants = [{"QX_HOT": "0"}, {"QX_HOT": "1", "QX_LANES": "1", "QX_MERGED": "1"}, {"QX_HOT": "1", "QX_LANES": "1", "QX_MERGED": "0"},
                {"QX_HOT": "1", "QX_LANES": "4", "QX_MERGED": "1"}, paired4,
                {"QX_HOT": "1", "QX_LANES": "2", "QX_MERGED": "1"}, {"QX_HOT": "1", "QX_LANES": "2", "QX_MERGED": "0"},
                {**paired4, "QX_MERGED": "1", "QX_PAIRED_RESET": "0"}, {**paired4, "QX_PAIRED_RESET": "0"},
                {**paired4, "QX_SHAPE": "0"}, {**paired4, "QX_SHAPE": "3"}, {**paired4, "QX_SHAPE": "5"}, {**paired4, "QX_PDL": "0"},
                {**paired4, "QX_STREAM_STORES": "1"}, {**paired4, "QX_STREAM_STORES": "2"}]
    queue_lengths = set()

    def run(var, bf16=False):
        for k_ in ("QX_HOT", "QX_LANES", "QX_MERGED", "QX_PAIRED_RESET", "QX_SHAPE", "QX_PDL", "QX_STREAM_STORES"):
            monkeypatch.delenv(k_, raising=False)
        for k_, v_ in {"QX_LANES": "1", "QX_MERGED": "1", **var}.items():
            monkeypatch.setenv(k_, v_)
        sim = pkg.QuadXSim(n, pkg.default_config(), seed=5)  # floor start, idle steps, auto-reset, noise
        d = sim.device
        # bf16: the policy's input buffer, row stride 32; the kernels write the first 20 columns
        obs = torch.zeros(steps, n, 32, device=d, dtype=torch.bfloat16)[..., :20] if bf16 else torch.zeros(steps, n, 20, device=d)
        tobs = torch.zeros(steps, n, 20, device=d); rew = torch.zeros(steps, n, device=d)
        te = torch.zeros(steps, n, dtype=torch.uint8, device=d); tr = torch.zeros(steps, n, dtype=torch.uint8, device=d)
        o0 = torch.zeros(n, 20, device=d)
        sim.reset(o0)
        for k in range(steps):
            sim.step_begin(acts[k], obs[k], rew[k], te[k], tr[k], tobs[k])
            torch.cuda.synchronize()
            queue_lengths.add(check_done_queue(sim, (te[k] | tr[k]).bool().cpu().numpy())[0])
            sim.step_end(obs[k])
        torch.cuda.synchronize()
        out = (obs, tobs, rew, te, tr, sim.get_state(), sim.episode_stats())
        sim.close()
        return out

    for generic in (False, True):
        if generic:
            monkeypatch.setenv("QX_FORCE_GENERIC", "1")
        o1, t1, r1, te1, tr1, s1, e1 = run(variants[0])
        assert int(te1.sum()) > n // 2  # episodes ended (floor rule) and restarted
        for var in variants[1:]:
            o2, t2, r2, te2, tr2, s2, e2 = run(var)
            assert torch.equal(te1, te2) and torch.equal(tr1, tr2) and e1[1:] == e2[1:], var
            assert torch.equal(o1.view(torch.int32), o2.view(torch.int32)), (var, float((o1 - o2).abs().max()))
            assert torch.equal(t1.view(torch.int32), t2.view(torch.int32)), (var, float((t1 - t2).abs().max()))
            assert torch.equal(r1.view(torch.int32), r2.view(torch.int32)), (var, float((r1 - r2).abs().max()))
            for k in s1:
                assert np.array_equal(s1[k].view(np.uint32), s2[k].view(np.uint32)), (var, k)
            del o2, t2
        for var in (paired4, {**paired4, "QX_PAIRED_RESET": "0"}):
            ob = run(var, bf16=True)[0]
            assert torch.equal(ob.view(torch.int16), o1.to(torch.bfloat16).view(torch.int16)), var
            assert torch.all(ob.as_strided((steps, n, 12), (n * 32, 32, 1), 20) == 0), var
    print(f"done-queue lengths seen over the variants: {len(queue_lengths)} distinct, max {max(queue_lengths)} of {n} envs")
    assert 0 in queue_lengths and len(queue_lengths) > 3
