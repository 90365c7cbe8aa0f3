#!/usr/bin/env python
"""Counterpart of the reference's simulation/train_hover.py:36-63 on the B200 path.

    python train_hover_b200.py --envs 16384 --steps 64 --iters 200
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 train_hover_b200.py --envs 131072

What the reference script does -> here:
  make_vec_env(QuadXHoverEnv, 16, SubprocVecEnv)  -> one batched sim per GPU (env ids sharded by rank)
  VecNormalize(norm_obs, norm_reward)             -> on-device running statistics (kernels K4)
  SAC/PPO("MlpPolicy", net_arch=[128,128], lr 3e-4) -> PPO, same network, rollout on tensor cores (K2) + GAE (K3)
  CheckpointCallback(min 20 000 steps, name with loss/len/rew) -> same cadence and file naming, torch .pt files
  tensorboard_log="./tensorboard"                 -> same tags (rollout/ep_len_mean, rollout/ep_rew_mean, time/fps, train/*)
  model.save("hover"); env.save("hover")          -> hover.pt (policy + optimiser + normalisation statistics)
  EvalCallback (SB3; not in the reference script) -> --eval-every K: deterministic evaluation on the device (ppo.PolicyEvaluator),
                                                     eval/mean_reward, eval/mean_ep_length, eval/success_rate
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=16384, help="envs per GPU (train_hover.py:41 uses 16 processes)")
    ap.add_argument("--steps", type=int, default=64, help="rollout length n_steps")
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--total-timesteps", type=int, default=0, help="stop after this many env steps (train_hover.py:60: 2 000 000)")
    ap.add_argument("--epochs", type=int, default=4)
    ap.add_argument("--batch", type=int, default=32768)
    ap.add_argument("--lr", type=float, default=3e-4)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--ent-coef", type=float, default=0.0)
    ap.add_argument("--gamma", type=float, default=0.99)
    ap.add_argument("--print-every", type=int, default=1)
    ap.add_argument("--target-kl", type=float, default=0.02)
    ap.add_argument("--log-std-init", type=float, default=-1.0)
    ap.add_argument("--save-path", default="./ppo_hover_checkpoints/")
    ap.add_argument("--min-steps-between-checkpoints", type=int, default=20000)  # train_hover.py:9
    ap.add_argument("--tensorboard", default="")
    ap.add_argument("--target-len", type=float, default=0.0, help="stop when rollout/ep_len_mean reaches this")
    ap.add_argument("--target-rew", type=float, default=0.0, help="... and rollout/ep_rew_mean reaches this (SURVEY C5: 181)")
    ap.add_argument("--gae-lambda", type=float, default=0.95)
    ap.add_argument("--lr-final-frac", type=float, default=1.0, help="linear learning-rate decay to this fraction ...")
    ap.add_argument("--lr-anneal-iters", type=int, default=0, help="... over this many iterations (0 = constant)")
    ap.add_argument("--log-std-min", type=float, default=None, help="floor under log_std while exploring ...")
    ap.add_argument("--log-std-min-final", type=float, default=None, help="... released linearly to this value ...")
    ap.add_argument("--log-std-min-iters", type=int, nargs=2, default=(0, 0), help="... between these iterations")
    ap.add_argument("--json", default="", help="write the per-iteration log here")
    ap.add_argument("--eval-every", type=int, default=0, help="evaluate the deterministic policy every K iterations and after training "
                                                                 "(EvalCallback; rank 0 only; 0 = off)")
    ap.add_argument("--eval-episodes", type=int, default=4096, help="episodes per evaluation (one env each)")
    ap.add_argument("--eval-seed", type=int, default=None, help="seed of the evaluation envs (default: --seed + 1)")
    args = ap.parse_args()
    eval_seed = args.seed + 1 if args.eval_seed is None else args.eval_seed

    import torch
    import torch.distributed as dist

    import __graft_entry__ as ge

    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    from fpv_drone_rl_agent_b200 import ppo

    cfg = ppo.PPOConfig(n_envs=args.envs, n_steps=args.steps, n_epochs=args.epochs, batch_size=args.batch, learning_rate=args.lr, seed=args.seed,
                        ent_coef=args.ent_coef, gamma=args.gamma, target_kl=args.target_kl, log_std_init=args.log_std_init, gae_lambda=args.gae_lambda,
                        lr_final_frac=args.lr_final_frac, lr_anneal_iters=args.lr_anneal_iters, log_std_min=args.log_std_min,
                        log_std_min_final=args.log_std_min_final, log_std_min_iters=tuple(args.log_std_min_iters))
    trainer = ppo.PPOTrainer(cfg, device=f"cuda:{local}", rank=rank, world=world)
    writer = None
    if args.tensorboard and rank == 0:
        from torch.utils.tensorboard import SummaryWriter

        writer = SummaryWriter(args.tensorboard)
    if rank == 0:
        os.makedirs(args.save_path, exist_ok=True)
    last_ckpt, log, t0, eval_s = 0, [], time.time(), 0.0

    def evaluate(out):
        """EvalCallback: the deterministic policy on its own envs; the summary goes into this iteration's log entry"""
        nonlocal eval_s
        te = time.time()
        ev, _ = trainer.evaluate(args.eval_episodes, eval_seed)
        eval_s += time.time() - te  # kept out of wall_s / fps, which stay the training rate
        out["eval"] = ev
        print(f"eval {out['timesteps']:>12,d} steps: mean_reward {ev['mean_reward']:9.2f} +/- {ev['std_reward']:.2f} mean_ep_length {ev['mean_ep_length']:7.1f} "
              f"success {ev['success_rate']:.3f} floor {ev['floor_rate']:.3f} oob {ev['oob_rate']:.3f} ({ev['n_episodes']} episodes)", flush=True)
        if writer:
            for tag, key in (("eval/mean_reward", "mean_reward"), ("eval/mean_ep_length", "mean_ep_length"), ("eval/success_rate", "success_rate")):
                writer.add_scalar(tag, ev[key], out["timesteps"])

    for it in range(args.iters):
        out = trainer.learn_iteration()
        torch.cuda.synchronize()
        out["wall_s"] = time.time() - t0 - eval_s
        out["fps"] = out["timesteps"] / out["wall_s"]
        if rank == 0:
            if it % args.print_every == 0:
                print(f"iter {it:4d} steps {out['timesteps']:>12,d} fps {out['fps']:>12,.0f} ep_len {out['ep_len_mean']:7.1f} ep_rew {out['ep_rew_mean']:9.2f} "
                      f"pg {out['pg']:+.4f} vf {out['vf']:.4f} kl {out['kl']:+.4f}", flush=True)
            log.append(out)
            if writer:
                for tag, key in (("rollout/ep_len_mean", "ep_len_mean"), ("rollout/ep_rew_mean", "ep_rew_mean"), ("time/fps", "fps"),
                                 ("train/policy_gradient_loss", "pg"), ("train/value_loss", "vf"), ("train/approx_kl", "kl"), ("train/clip_fraction", "clipfrac")):
                    writer.add_scalar(tag, out[key], out["timesteps"])
            if args.eval_every and (it + 1) % args.eval_every == 0:
                evaluate(out)
            if out["timesteps"] - last_ckpt >= args.min_steps_between_checkpoints:  # train_hover.py:17-31
                name = f"ppo_hover_{out['timesteps']}_steps_{round(out['vf'], 2)}_len{round(out['ep_len_mean'], 2)}_rew{round(out['ep_rew_mean'], 2)}.pt"
                trainer.save(os.path.join(args.save_path, name))
                last_ckpt = out["timesteps"]
        if args.target_len and out["ep_len_mean"] >= args.target_len and (not args.target_rew or out["ep_rew_mean"] >= args.target_rew):
            break
        if args.total_timesteps and out["timesteps"] >= args.total_timesteps:
            break
    if rank == 0:
        if args.eval_every and log and "eval" not in log[-1]:  # the trained policy (an evaluation of the same weights would repeat itself)
            evaluate(log[-1])
        trainer.save("hover.pt")  # train_hover.py:62-63
        trainer.save_sb3("hover_sb3.zip")  # policy.pth under SB3's parameter names + VecNormalize statistics (ppo.export_sb3_zip)
        if args.json:
            json.dump(log, open(args.json, "w"))
        print("Training complete.")
    if world > 1:
        # the captured graphs hold NCCL kernels: release them before the communicator goes away
        trainer._epoch_graph = None
        trainer.rollout._graph = None
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
