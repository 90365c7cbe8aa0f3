"""qx_render / QuadXSim.render / QuadXHoverEnv(render_mode="rgb_array"): the FPV camera frame drawn on the device.

The frame is drawn from the same row spans vision_raster (vision_mode = 1) counts, so the reference's detect_rectangle
(hover.py:157-222) run on a device frame must report exactly the camera columns of the observation taken at that pose.
Poses are placed as in tests/test_gpu_parity.py: aviary_steps_per_step = 0, qx_set_state, one step -- the step runs no
physics, so the observation and the frame come from exactly the pose that was set."""
import os
import re

import numpy as np
import pytest
import torch

HOVER_THR = float(np.sqrt(0.1 * 9.81 / 4.0))  # pwm at which thrust = weight (cf2x.yaml:2, cf2x.urdf:10)
RED, SKY = np.array([200, 0, 0, 255], np.uint8), np.array([170, 190, 230, 255], np.uint8)


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge

    ge.build()
    import fpv_drone_rl_agent_b200 as pkg

    return pkg


def _bufs(sim):
    n, d = sim.n, sim.device
    return (torch.zeros(n, 20, device=d), torch.zeros(n, device=d), torch.zeros(n, dtype=torch.uint8, device=d),
            torch.zeros(n, dtype=torch.uint8, device=d))


def _posed(pkg, pos, quat, **cfg_kw):
    """A sim whose env i sits at (pos[i], quat[i]) (float32), its observation of that pose, and the pose as stored."""
    n = pos.shape[0]
    cfg = pkg.default_config()
    cfg.update(start_pos=[0, 0, 1.2], reset_idle_steps=0, auto_reset=0, noise=0, vision_mode=1, aviary_steps_per_step=0, max_steps=10000)
    cfg.update(**cfg_kw)
    sim = pkg.QuadXSim(n, cfg, seed=78)
    obs, rew, te, tr = _bufs(sim)
    sim.reset(obs)
    st = sim.get_state()
    for j, key in enumerate(("px", "py", "pz")):
        st[key] = pos[:, j].astype(np.float32)
    for j, key in enumerate(("qx", "qy", "qz", "qw")):
        st[key] = quat[:, j].astype(np.float32)
    sim.set_state(st)
    sim.step(torch.zeros(n, 4, device=sim.device), obs, rew, te, tr)
    st2 = sim.get_state()
    pos2 = np.stack([st2["px"], st2["py"], st2["pz"]], 1).astype(np.float64)
    quat2 = np.stack([st2["qx"], st2["qy"], st2["qz"], st2["qw"]], 1).astype(np.float64)
    assert np.array_equal(pos2.astype(np.float32), pos.astype(np.float32))
    return sim, obs.cpu().numpy(), pos2, quat2


def _dome_poses(n, seed):
    from oracle.quadx_model import euler_to_quat

    rng = np.random.default_rng(seed)
    pos = rng.uniform(-1.8, 1.8, (n, 3))
    pos[:, 2] = rng.uniform(0.3, 2.4, n)
    return pos, euler_to_quat(rng.uniform(-0.4, 0.4, (n, 3)))


def _corner_depths(pos, quat, p):
    from oracle import vision

    eye, fwd, _, _ = vision.camera_frame(pos, quat, p)
    return np.einsum("nmj,nj->nm", vision.panel_box_corners()[None] - eye[:, None], fwd)


def _red(img):
    return (img[..., 0] > 100) & (img[..., 1] == 0) & (img[..., 2] == 0)


def _boundary(red):
    """red pixels with a non-red 4-neighbour (outside the image counts as non-red)"""
    p = np.pad(red, 1)
    return red & ~(p[:-2, 1:-1] & p[2:, 1:-1] & p[1:-1, :-2] & p[1:-1, 2:])


def _compare_frames(dev, ref):
    """-> number of differing pixels; asserts that each is on the red region's boundary in the image where it is red and
    that every pixel is one of the two colours"""
    assert np.all(np.all(dev == RED, -1) | np.all(dev == SKY, -1))
    rd, rr = _red(dev), _red(ref)
    diff = rd != rr
    assert not (diff & ~(_boundary(rd) | _boundary(rr))).any()
    return int(diff.sum())


def _detector_reason(img):
    """detect_rectangle (hover.py:157-222) step by step: (reason it rejects the frame or "ok", bounding box w, h)"""
    import cv2

    red = _red(img).astype(np.uint8) * 255
    if not red.any():
        return "no red", 0, 0
    if red[0, :].any() or red[-1, :].any() or red[:, 0].any() or red[:, -1].any():
        return "at edge", 0, 0
    contours, _ = cv2.findContours(red, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
    contour = max(contours, key=cv2.contourArea)
    _, _, bw, bh = cv2.boundingRect(contour)
    approx = cv2.approxPolyDP(contour, 0.04 * cv2.arcLength(contour, True), True)
    return ("ok" if len(approx) == 4 else f"approxPolyDP {len(approx)} vertices"), bw, bh


def _same_ratio(r32, kernel):
    """The kernel's bounding-box ratio is w * rcp(h) (the library builds with --use_fast_math): within 2 ulp of the rounded
    w / h.  Distinct ratios of integers <= 128 lie >= 6e-5 apart, so this still means the same bounding box."""
    return bool(np.all(np.abs(r32.astype(np.float64) - kernel.astype(np.float64)) <= 2 * np.spacing(np.abs(r32))))


def _features_agree(frames, obs, what):
    """detect_rectangle on the device frames against the observation's camera columns (7:9 centre, 11 area, 13 visible,
    14 ratio).  Returns (frames both see, visibility mismatches by reason)."""
    from oracle.hover_oracle import detect_rectangle

    n = frames.shape[0]
    V, C, A, R = np.zeros(n, bool), np.zeros((n, 2)), np.zeros(n), np.zeros(n)
    for i in range(n):
        V[i], C[i], A[i], R[i] = detect_rectangle(frames[i])
    vis = obs[:, 13] > 0.5
    reasons = {}
    for i in np.nonzero(vis != V)[0]:
        why, bw, bh = _detector_reason(frames[i])
        if vis[i]:  # the kernel sees a box the detector rejects: only its 4-vertex test may do that
            assert why.startswith("approxPolyDP"), (what, i, why)
        else:  # the detector takes a box the kernel rejects: only the kernel's 2-px bounding-box floor may do that
            assert why == "ok" and (bw < 2 or bh < 2), (what, i, why, bw, bh)
            why = "bounding box under 2 px"
        reasons[why] = reasons.get(why, 0) + 1
    both = vis & V
    # vision_raster's area is Pick's theorem over the spans (N - B/2 - 1), which holds for a simple contour; where the silhouette
    # ends in a one-pixel spike, cv2's contour runs through that pixel twice and contourArea is 0.5 px^2 smaller per such pixel
    spikes = 0
    for i in np.nonzero(both & (A != obs[:, 11].astype(np.float64)))[0]:
        rep = _repeated_contour_pixels(frames[i])
        assert rep > 0 and (obs[i, 11] - A[i]) * frames.shape[1] ** 2 == 0.5 * rep, (what, i, rep, (obs[i, 11] - A[i]) * frames.shape[1] ** 2)
        spikes += 1
    r32 = R[both].astype(np.float32)
    assert _same_ratio(r32, obs[both, 14]), (what, np.abs(R - obs[:, 14])[both].max())
    worst_c = float(np.abs(obs[:, 7:9] - C)[both].max() * 64) if both.any() else 0.0
    print(f"{what}: {n} frames, both see the panel in {int(both.sum())}, bounding box differs in 0 (ratio bit-equal in "
          f"{int((r32 == obs[both, 14]).sum())}), area in 0 but {spikes} with a one-pixel spike, worst centre error {worst_c:.2f} px, visibility mismatches {int((vis != V).sum())} {reasons}")
    # the centre is vision_raster's stand-in (mean of the projected front-face corners), computed without the pixels, so the frame
    # cannot move it: held to the project's bound of that stand-in against the detector (1.5 px, tests/test_oracle_golden.py);
    # flown frames reach ~1.0 px
    assert worst_c <= 1.5, (what, worst_c)
    return int(both.sum()), reasons


def _repeated_contour_pixels(img):
    """pixels the detector's contour (the largest external one) passes more than once"""
    import cv2

    cs, _ = cv2.findContours(_red(img).astype(np.uint8) * 255, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_NONE)
    c = max(cs, key=cv2.contourArea).reshape(-1, 2)
    return len(c) - len({tuple(x) for x in c})


@pytest.mark.gpu
def test_frames_equal_cpu_rasteriser(pkg):
    """RGBA frames of 512 in-dome poses (every corner in front) against oracle.vision.render_rgba of the same float32 pose:
    a pixel may differ only on the red region's boundary (fp32 vs float64), in at most 1 % of the frames."""
    from oracle import vision
    from oracle.quadx_model import QuadXParams

    p = QuadXParams()
    n = 512
    pos, quat = _dome_poses(n, 3)
    sim, obs, pos2, quat2 = _posed(pkg, pos, quat)
    assert (_corner_depths(pos2, quat2, p) > p.cam_near).all()
    frames = sim.render().cpu().numpy()
    assert frames.shape == (n, 128, 128, 4) and frames.dtype == np.uint8
    px_diff = [_compare_frames(frames[i], vision.render_rgba(pos2[i], quat2[i], p)) for i in range(n)]
    n_frames = sum(d > 0 for d in px_diff)
    print(f"device vs CPU rasteriser: {n} frames, {n_frames} with a differing pixel, {sum(px_diff)} differing pixels, "
          f"{int(_red(frames).any(axis=(1, 2)).sum())} frames show the box")
    assert _red(frames).any(axis=(1, 2)).sum() > n // 2
    assert n_frames <= 0.01 * n
    sim.close()


@pytest.mark.gpu
def test_frames_give_raster_features_exactly(pkg):
    """The reference's detector on device frames reports vision_mode = 1's features: on random poses and on frames of a flown
    rollout (4 096 envs, noise, auto-reset) taken at steps that include resets.  Wherever both see the panel: bounding box equal
    (no flips), area equal except 0.5 px^2 per pixel the detector's contour passes twice (a one-pixel spike, where the Pick's-
    theorem area of vision_raster does not hold), centre within the 1.5 px of its stand-in.  A visibility mismatch only where approxPolyDP does not
    find 4 vertices or the bounding box is under 2 px."""
    pos, quat = _dome_poses(512, 11)
    sim, obs, _, _ = _posed(pkg, pos, quat)
    seen, _ = _features_agree(sim.render().cpu().numpy(), obs, "random poses")
    assert seen > 250
    sim.close()

    n = 4096
    cfg = pkg.default_config()
    cfg.update(vision_mode=1, auto_reset=1, noise=1, start_pos=[0, 0, 1.0], spawn_throttle=HOVER_THR, reset_idle_steps=0,
               spawn_pos_noise=0.6, spawn_yaw_noise=0.4, max_steps=24)
    sim = pkg.QuadXSim(n, cfg, seed=5)
    obs, rew, te, tr = _bufs(sim)
    sim.reset(obs)
    rng = np.random.default_rng(9)
    taken, resets = 0, 0
    for k in range(30):
        a = rng.uniform(-1, 1, (n, 4)).astype(np.float32)
        a[:, :3] *= 0.3
        a[:, 3] = 0.15 * a[:, 3]  # around the hover throttle ((a3 + 1) / 2 ~ 0.495)
        sim.step(torch.as_tensor(a, device=sim.device), obs, rew, te, tr)
        if k in (3, 11, 18, 23, 24, 29):
            frames = sim.render().cpu().numpy()
            done = int((te | tr).sum().item())
            resets += done
            s, _ = _features_agree(frames, obs.cpu().numpy(), f"rollout step {k + 1} ({done} envs reset in it)")
            taken += s
    assert resets > 0 and taken > n
    sim.close()


def _yawed_across_panel(n, seed):
    """poses next to the panel, yawed 60-120 deg, so that the box crosses the camera plane"""
    from oracle.quadx_model import euler_to_quat

    rng = np.random.default_rng(seed)
    pos = np.stack([rng.uniform(3.6, 4.5, n), rng.uniform(-1.2, 1.2, n), rng.uniform(5.2, 6.8, n)], 1)
    e = rng.uniform(-0.2, 0.2, (n, 3))
    e[:, 2] = rng.choice([-1.0, 1.0], n) * np.deg2rad(rng.uniform(60, 120, n))
    return pos, euler_to_quat(e)


def _render_rgba_clipped(pos, quat, p):
    """oracle.vision.render_rgba for a box that may cross the camera's near plane (a drone yawed across the panel): the box is
    clipped to depth > cam_near first, so the silhouette is the convex hull of the projected corners in front of the plane and
    of the points where the box edges cross it.  Float64 throughout (the hull is found on the float64 points)."""
    from oracle import vision

    corners = vision.panel_box_corners()
    eye, fwd, right, up = vision.camera_frame(pos[None], quat[None], p)
    depth = (corners - eye[0]) @ fwd[0]
    res = p.cam_res
    img = np.empty((res, res, 4), np.uint8)
    img[...] = SKY
    front = depth > p.cam_near
    pts = [corners[k] for k in range(8) if front[k]]
    for a, b in vision.BOX_EDGES:
        if front[a] != front[b]:
            t = (p.cam_near - depth[a]) / (depth[b] - depth[a])
            pts.append(corners[a] + t * (corners[b] - corners[a]))
    if not pts:
        return img
    px, py, _ = vision.project(np.array(pts), eye, fwd, right, up, p)
    xy = np.stack([px[0], py[0]], axis=1)
    # hull: monotone chain on the float64 points, counter-clockwise in (x, y)
    order = sorted(range(len(xy)), key=lambda i: (xy[i, 0], xy[i, 1]))

    def cross(o, a, b):
        return (xy[a, 0] - xy[o, 0]) * (xy[b, 1] - xy[o, 1]) - (xy[a, 1] - xy[o, 1]) * (xy[b, 0] - xy[o, 0])

    lower, upper = [], []
    for i in order:
        while len(lower) >= 2 and cross(lower[-2], lower[-1], i) <= 0:
            lower.pop()
        lower.append(i)
    for i in reversed(order):
        while len(upper) >= 2 and cross(upper[-2], upper[-1], i) <= 0:
            upper.pop()
        upper.append(i)
    hull = xy[lower[:-1] + upper[:-1]]
    ys, xs = np.mgrid[0:res, 0:res]
    cx, cy = xs + 0.5, ys + 0.5
    red = np.ones((res, res), bool)
    m = hull.shape[0]
    for i in range(m):
        x0, y0 = hull[i]
        x1, y1 = hull[(i + 1) % m]
        red &= (x1 - x0) * (cy - y0) - (y1 - y0) * (cx - x0) >= 0
    img[red] = RED
    return img


@pytest.mark.gpu
def test_near_plane_clipping(pkg):
    """Boxes crossing the near plane are clipped to it: frames against a float64 clipped rasteriser (boundary pixels only,
    in at most 2 % of the frames).  vision_mode = 1 reports these poses unseen, and so does the detector on the frame."""
    from oracle import vision
    from oracle.hover_oracle import detect_rectangle
    from oracle.quadx_model import QuadXParams

    p = QuadXParams()
    pos, quat = _yawed_across_panel(512, 21)
    sim, obs, pos2, quat2 = _posed(pkg, pos, quat)
    dep = _corner_depths(pos2, quat2, p)
    cross = (dep <= p.cam_near).any(1) & (dep > p.cam_near).any(1)
    frames = sim.render().cpu().numpy()
    px_diff, shown = [], 0
    for i in np.nonzero(cross)[0]:
        ref = _render_rgba_clipped(pos2[i], quat2[i], p)
        px_diff.append(_compare_frames(frames[i], ref))
        shown += bool(_red(frames[i]).any())
        assert obs[i, 13] == 0.0 and not detect_rectangle(frames[i])[0]
    n_frames = sum(d > 0 for d in px_diff)
    print(f"near-plane clipping: {int(cross.sum())} poses cross the camera plane, {shown} of them show part of the box, "
          f"{n_frames} frames with a differing pixel ({sum(px_diff)} pixels)")
    assert cross.sum() >= 200 and shown >= 100
    assert n_frames <= 0.02 * cross.sum()
    sim.close()


@pytest.mark.gpu
def test_subsets_formats_and_graph(pkg):
    """n = 1 000 (not a multiple of 32): a ragged env_idx with duplicates and out-of-range entries gives the matching frames
    of the full render (background where out of range); MASK = 255 * the red mask of RGBA; m = 1; qx_step + qx_render
    captured in a CUDA graph and replayed draws what the eager calls draw."""
    n = 1000
    pos, quat = _dome_poses(n, 31)
    sim, _, _, _ = _posed(pkg, pos, quat)
    full = sim.render()
    mask = sim.render(fmt="mask")
    assert mask.shape == (n, 128, 128)
    assert torch.equal(mask, 255 * ((full[..., 0] > 100) & (full[..., 1] == 0) & (full[..., 2] == 0)).to(torch.uint8))
    idx = [5, 999, 5, -1, 1000, 0, 123, 123, 2**31 - 1, 500, 998, 1, -(2**31), 77, 5, 640, 641]
    sub = sim.render(idx)
    sub_t = sim.render(torch.tensor(idx, dtype=torch.int32, device=sim.device), fmt="mask")
    sky = torch.tensor(SKY, device=sim.device).expand(128, 128, 4)
    for j, i in enumerate(idx):
        if 0 <= i < n:
            assert torch.equal(sub[j], full[i]) and torch.equal(sub_t[j], mask[i]), (j, i)
        else:
            assert torch.equal(sub[j], sky) and not sub_t[j].any(), (j, i)
    out = torch.full((1, 128, 128, 4), 7, dtype=torch.uint8, device=sim.device)
    assert sim.render([321], out=out) is out and torch.equal(out[0], full[321])
    sim.close()

    def make():
        cfg = pkg.default_config()
        cfg.update(vision_mode=1, start_pos=[0, 0, 1.0], spawn_throttle=HOVER_THR, reset_idle_steps=0, spawn_pos_noise=0.6,
                   spawn_yaw_noise=0.4, max_steps=6)
        s = pkg.QuadXSim(n, cfg, seed=17)
        b = _bufs(s)
        s.reset(b[0])
        return s, b

    (eager, be), (graphed, bg) = make(), make()
    act = torch.empty(n, 4, device=eager.device)
    frames_g = torch.empty(n, 128, 128, 4, dtype=torch.uint8, device=eager.device)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        graphed.step(act, *bg)
        graphed.render(out=frames_g)
    gen = torch.Generator(device=eager.device).manual_seed(0)
    for k in range(10):
        act.copy_(0.2 * torch.rand(n, 4, device=eager.device, generator=gen) - 0.1)
        eager.step(act, *be)
        frames_e = eager.render()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(be[0], bg[0]) and torch.equal(frames_e, frames_g), k
    eager.close()
    graphed.close()


@pytest.mark.gpu
def test_facade_rgb_array(pkg):
    """QuadXHoverEnv(render_mode="rgb_array"): render() after reset and after a step is the uint8 frame of that state, and the
    reference's detector on it reports the observation's camera columns.  Without render_mode it still raises."""
    from oracle.hover_oracle import detect_rectangle

    assert pkg.QuadXHoverEnv.metadata["render_modes"] == ["rgb_array"]
    env = pkg.QuadXHoverEnv(render_mode="rgb_array", vision_mode=1)
    obs, _ = env.reset()
    for k in range(3):
        img = env.render()
        assert img.shape == (128, 128, 4) and img.dtype == np.uint8
        v, c, a, r = detect_rectangle(img)
        assert v == (obs[13] > 0.5) and v, k
        assert a == obs[11] and _same_ratio(np.float32([r]), np.float32([obs[14]])) and np.abs(c - obs[7:9]).max() * 64 <= 1.5, k
        obs, *_ = env.step(np.array([0.0, 0.0, 0.0, 0.2]))
    env.close()
    env = pkg.QuadXHoverEnv()
    env.reset()
    with pytest.raises(NotImplementedError, match="out of scope"):
        env.render()
    env.close()


@pytest.mark.gpu
def test_invalid_arguments(pkg):
    """Every rejected call of qx_render names its reason and launches nothing; m = 0 is a no-op."""
    import ctypes as C

    from fpv_drone_rl_agent_b200 import _lib

    L = _lib.lib()
    sim = pkg.QuadXSim(64)
    buf = torch.empty(64, 128, 128, 4, dtype=torch.uint8, device=sim.device)
    idx = torch.zeros(4, dtype=torch.int32, device=sim.device)
    s = sim._stream()
    ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    cases = [
        (lambda: L.qx_render(sim._h, None, 64, 2, ptr(buf), s), "fmt is QX_FRAME_RGBA or QX_FRAME_MASK"),
        (lambda: L.qx_render(sim._h, ptr(idx), -1, 0, ptr(buf), s), "m < 0"),
        (lambda: L.qx_render(sim._h, None, 63, 0, ptr(buf), s), "m must equal n_envs"),
        (lambda: L.qx_render(sim._h, ptr(idx), 4, 1, None, s), "null frames_dev"),
        (lambda: L.qx_render(sim._h, ptr(idx), 4, 1, C.c_void_p(buf.data_ptr() + 4), s), "16-byte aligned"),
    ]
    yaw = pkg.QuadXSim(64, task=pkg.QX_TASK_YAW)
    cases.append((lambda: L.qx_render(yaw._h, None, 64, 0, ptr(buf), s), "hover task only"))
    cfg = pkg.default_config()
    cfg.update(cam_res=126.0)
    odd = pkg.QuadXSim(64, cfg)
    cases.append((lambda: L.qx_render(odd._h, None, 64, 0, ptr(buf), s), "positive multiple of 4"))
    for call, msg in cases:
        before = L.qx_launch_count()
        with pytest.raises(pkg.QxError, match=msg):
            _lib.check(call())
        assert L.qx_launch_count() == before, msg
    before = L.qx_launch_count()
    assert L.qx_render(sim._h, ptr(idx), 0, 0, None, s) == 0 and L.qx_launch_count() == before
    with pytest.raises(pkg.QxError, match="hover task only"):
        yaw.render()
    with pytest.raises(ValueError):
        sim.render(fmt="bgr")
    for x in (sim, yaw, odd):
        x.close()


def test_render_kernel_does_not_spill():
    """CPU: both instantiations of the frame kernel compile without spills (ptxas -v in csrc/build.log)."""
    import __graft_entry__ as ge

    ge.build()
    from fpv_drone_rl_agent_b200 import _lib

    log = os.path.join(os.path.dirname(_lib.LIB_PATH), "build.log")
    if not os.path.exists(log):  # library was already up to date and the log is not in the checkout: rebuild once
        import importlib.util

        spec = importlib.util.spec_from_file_location("qx_build", os.path.join(os.path.dirname(_lib.LIB_PATH), "build.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.build(force=True)
    text = open(log).read()
    found = re.findall(r"Compiling entry function '(\S*render_kernel\S*)' for 'sm_100a'.*?(\d+) bytes stack frame, (\d+) bytes spill stores, "
                       r"(\d+) bytes spill loads.*?Used (\d+) registers", text, re.S)
    assert len(found) == 2, found
    for name, stack, st, ld, regs in found:
        assert int(st) == 0 and int(ld) == 0 and int(stack) == 0, (name, stack, st, ld)
        assert int(regs) <= 64, (name, regs)  # 4 blocks of 256 threads per SM
