"""qx_render (K6, the FPV camera frame) on the GPU: kernel time, frames/s and bytes written per second for m = 4 096,
16 384 and 65 536 frames in both formats, and the per-step cost of a 16 384-env pixel-observation loop (qx_step +
qx_render(MASK) against qx_step alone).

    python tools/render_bench.py [--reps 30] [--json out.json]

Bytes = m * res^2 * channels written by the kernel (it reads 32 B of state per frame); the fraction is of 6 538.6 GB/s, the
HBM rate the project divides by (DESIGN 7).  Times are CUDA-event means over `reps` back-to-back launches after a warm-up;
every output buffer but the 4 096-frame mask (67 MB) is larger than the 126 MB L2.  The card's name and power limit are read
in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_GBS = 6538.6


def timed(fn, reps, rounds=5):
    """median over `rounds` of the mean time of `reps` back-to-back calls, in microseconds"""
    import torch

    ts = []
    for _ in range(rounds):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            fn()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e) * 1e3 / reps)
    return statistics.median(ts)


def flown_sim(pkg, n, seed=1):
    """n envs after a few steps of random flight from spread-out spawns, so that the frames differ"""
    import numpy as np
    import torch

    cfg = pkg.default_config()
    cfg.update(start_pos=[0, 0, 1.0], spawn_throttle=0.495, reset_idle_steps=0, spawn_pos_noise=0.8, spawn_yaw_noise=0.4)
    sim = pkg.QuadXSim(n, cfg, seed=seed)
    d = sim.device
    bufs = (torch.zeros(n, 20, device=d), torch.zeros(n, device=d), torch.zeros(n, dtype=torch.uint8, device=d),
            torch.zeros(n, dtype=torch.uint8, device=d))
    sim.reset(bufs[0])
    rng = np.random.default_rng(seed)
    for _ in range(4):
        a = rng.uniform(-0.2, 0.2, (n, 4)).astype(np.float32)
        sim.step(torch.as_tensor(a, device=d), *bufs)
    torch.cuda.synchronize()
    return sim, bufs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--json", default=None, help="also write the results to this file")
    args = ap.parse_args()
    import torch

    import __graft_entry__ as ge

    ge.build()
    import fpv_drone_rl_agent_b200 as pkg
    from fpv_drone_rl_agent_b200 import _lib

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    card = card.splitlines()[torch.cuda.current_device()] if card else "unknown"
    print(f"card: {card}   library: {os.path.relpath(_lib.LIB_PATH, ROOT)}")
    res = 128
    rows = []
    for m in (4096, 16384, 65536):
        sim, _ = flown_sim(pkg, m)
        for fmt, ch in (("rgba", 4), ("mask", 1)):
            shape = (m, res, res, 4) if ch == 4 else (m, res, res)
            out = torch.empty(shape, dtype=torch.uint8, device=sim.device)
            for _ in range(3):
                sim.render(fmt=fmt, out=out)
            torch.cuda.synchronize()
            us = timed(lambda: sim.render(fmt=fmt, out=out), args.reps)
            nbytes = m * res * res * ch
            gbs = nbytes / (us * 1e-6) / 1e9
            red = float((out[..., 0] if ch == 4 else out).eq(200 if ch == 4 else 255).any(-1).any(-1).float().mean())
            rows.append(dict(frames=m, fmt=fmt, bytes=nbytes, us=us, frames_per_s=m / (us * 1e-6), gb_per_s=gbs, frac_hbm=gbs / HBM_GBS,
                             frames_showing_box=red))
            print(f"qx_render {fmt:4s} m={m:6d}: {us:9.1f} us  {m / (us * 1e-6) / 1e6:8.1f} Mframes/s  {nbytes / 1e6:8.1f} MB  "
                  f"{gbs:7.1f} GB/s = {gbs / HBM_GBS:.3f} of {HBM_GBS} GB/s   (box in {100 * red:.0f} % of the frames)")
            del out
        sim.close()
        torch.cuda.empty_cache()

    # pixel-observation loop: 16 384 envs, every step followed by the mask frame of every env
    n = 16384
    sim, bufs = flown_sim(pkg, n, seed=2)
    act = torch.zeros(n, 4, device=sim.device)
    mask = torch.empty(n, res, res, dtype=torch.uint8, device=sim.device)

    def step():
        sim.step(act, *bufs)

    def step_render():
        sim.step(act, *bufs)
        sim.render(fmt="mask", out=mask)

    def render_only():
        sim.render(fmt="mask", out=mask)

    for f in (step, step_render, render_only):
        for _ in range(5):
            f()
    torch.cuda.synchronize()
    t_step, t_both, t_mask = [], [], []
    for _ in range(3):  # alternated, so that a drift of the clock shows in both
        t_step.append(timed(step, args.reps, rounds=3))
        t_both.append(timed(step_render, args.reps, rounds=3))
        t_mask.append(timed(render_only, args.reps, rounds=3))
    loop = dict(envs=n, step_us=statistics.median(t_step), step_plus_mask_us=statistics.median(t_both), mask_alone_us=statistics.median(t_mask))
    loop["added_per_step_us"] = loop["step_plus_mask_us"] - loop["step_us"]
    print(f"pixel-observation loop, {n} envs: qx_step {loop['step_us']:.1f} us/step, qx_step + qx_render(MASK) {loop['step_plus_mask_us']:.1f} us/step "
          f"(+{loop['added_per_step_us']:.1f} us; the mask render alone {loop['mask_alone_us']:.1f} us)")
    sim.close()
    result = dict(card=card, library=os.path.relpath(_lib.LIB_PATH, ROOT), reps=args.reps, render=rows, pixel_loop=loop)
    print(json.dumps(result))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
