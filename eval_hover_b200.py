#!/usr/bin/env python
"""Counterpart of the reference's simulation/test_hover.py:7-27 on the B200 path: play a trained policy back.

    python eval_hover_b200.py --checkpoint hover.pt --episodes 4096 --seed 1 [--render]
    python eval_hover_b200.py --sb3-zip model.zip [--vecnormalize stats.npz] [--clip-obs 10] --episodes 4096 --seed 1

What the reference script does -> here:
  PPO.load("hover") + VecNormalize.load(..., training=False, norm_reward=False) -> the checkpoint of PPOTrainer.save (its policy,
                                                     observation statistics, clip_obs and net_arch)
  QuadXHoverEnv(render=True)                      -> --render: the floor rule off (hover.py:283)
  SAC.load("hover") / PPO.load("hover")            -> --sb3-zip: a stable-baselines3 archive (sac.load_sb3_zip; SAC actors run
                                                     on the K8 kernel, PPO policies on K2); --vecnormalize: its VecNormalize
                                                     statistics as .npz (tools/sb3_vecnormalize_to_npz.py converts the .pkl;
                                                     default: the archive's own vecnormalize.npz, if any, else none)
  model.predict(obs, deterministic=True) until done -> ppo.evaluate_policy: every env flies one episode on the device
Prints one JSON line: mean_reward, std_reward, mean_ep_length, success_rate, floor_rate, oob_rate, n_episodes, steps
(with --sb3-zip also "algorithm": "SAC" or "PPO").
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--checkpoint", default="hover.pt", help="a checkpoint written by PPOTrainer.save (train_hover_b200.py)")
    ap.add_argument("--sb3-zip", default=None, help="instead of --checkpoint: a stable-baselines3 SAC or PPO model archive (.zip)")
    ap.add_argument("--vecnormalize", default=None, help="with --sb3-zip: VecNormalize statistics (.npz, export_vecnormalize keys)")
    ap.add_argument("--clip-obs", type=float, default=None, help="with --sb3-zip: VecNormalize clip_obs (default: the statistics' own, else 10)")
    ap.add_argument("--episodes", type=int, default=4096, help="episodes, one env each")
    ap.add_argument("--seed", type=int, default=1, help="seed of the evaluation envs")
    ap.add_argument("--render", action="store_true", help="hover.py's render=True: the floor rule is off")
    ap.add_argument("--device", default="cuda:0")
    args = ap.parse_args()

    import torch

    import __graft_entry__ as ge

    ge.build()
    from fpv_drone_rl_agent_b200 import QX_TASK_HOVER, QX_TASK_YAW, default_config, ppo, sac

    dev = torch.device(args.device)
    if args.sb3_zip is not None:
        arc = sac.load_sb3_zip(args.sb3_zip, dev)
        obs_dim = arc.model.obs_dim
        task = {20: QX_TASK_HOVER, 12: QX_TASK_YAW}.get(obs_dim)
        if task is None:
            raise SystemExit(f"{args.sb3_zip}: a policy with {obs_dim} inputs is for neither task (hover 20, yaw 12)")
        vn = sac.load_vecnormalize(args.vecnormalize) if args.vecnormalize is not None else arc.vecnormalize
        stats = sac.obs_stats_from_vecnormalize(vn, dev) if vn is not None else None
        clip = args.clip_obs if args.clip_obs is not None else (float(vn["clip_obs"]) if vn is not None and "clip_obs" in vn else 10.0)
        env_cfg = default_config(task)
        env_cfg.update(render=int(args.render))
        summary, _ = ppo.evaluate_policy(arc.pack(dev), stats, env_cfg, args.episodes, args.seed, task=task, obs_clip=clip, device=dev)
        summary["algorithm"] = arc.algorithm
        print(json.dumps(summary), flush=True)
        return
    sd = torch.load(args.checkpoint, map_location=dev, weights_only=True)
    cfg = sd["cfg"]
    w1 = sd["model"]["pi1.weight"]
    obs_dim, act_dim = int(w1.shape[1]), int(sd["model"]["mu.weight"].shape[0])
    task = {20: QX_TASK_HOVER, 12: QX_TASK_YAW}.get(obs_dim)
    if task is None:
        raise SystemExit(f"{args.checkpoint}: a policy with {obs_dim} inputs is for neither task (hover 20, yaw 12)")
    model = ppo.ActorCritic(obs_dim, act_dim, hidden=int(cfg.get("net_arch", ppo.HID))).to(dev)
    with torch.no_grad():
        for k, v in model.state_dict().items():
            v.copy_(sd["model"][k])
    packed = ppo.PackedPolicy(model, dev)
    stats = None
    if cfg.get("norm_obs", True):
        stats = ppo.RunningStats(obs_dim, dev)
        stats.load_state_dict(sd["obs_stats"])
    env_cfg = default_config(task)
    env_cfg.update(render=int(args.render))
    summary, _ = ppo.evaluate_policy(packed, stats, env_cfg, args.episodes, args.seed, task=task, obs_clip=float(cfg.get("clip_obs", 10.0)),
                                     device=dev)
    print(json.dumps(summary), flush=True)


if __name__ == "__main__":
    main()
