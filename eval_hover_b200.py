#!/usr/bin/env python
"""Counterpart of the reference's simulation/test_hover.py:7-27 on the B200 path: play a trained policy back.

    python eval_hover_b200.py --checkpoint hover.pt --episodes 4096 --seed 1 [--render]

What the reference script does -> here:
  PPO.load("hover") + VecNormalize.load(..., training=False, norm_reward=False) -> the checkpoint of PPOTrainer.save (its policy,
                                                     observation statistics, clip_obs and net_arch)
  QuadXHoverEnv(render=True)                      -> --render: the floor rule off (hover.py:283)
  model.predict(obs, deterministic=True) until done -> ppo.evaluate_policy: every env flies one episode on the device
Prints one JSON line: mean_reward, std_reward, mean_ep_length, success_rate, floor_rate, oob_rate, n_episodes, steps.
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
    ap.add_argument("--episodes", type=int, default=4096, help="episodes, one env each")
    ap.add_argument("--seed", type=int, default=1, help="seed of the evaluation envs")
    ap.add_argument("--render", action="store_true", help="hover.py's render=True: the floor rule is off")
    ap.add_argument("--device", default="cuda:0")
    args = ap.parse_args()

    import torch

    import __graft_entry__ as ge

    ge.build()
    from fpv_drone_rl_agent_b200 import QX_TASK_HOVER, QX_TASK_YAW, default_config, ppo

    dev = torch.device(args.device)
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
