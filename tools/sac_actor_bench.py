"""SAC actor forward (K8, sac_actor_forward) and SAC policy evaluation on the GPU, next to the PPO forward (K2) they compare with.

  * kernel rate: CUDA-event time of `reps` launches captured in one graph (hover shape 20 -> 4, [128, 128]), the K8 and K2
    graphs alternated 5 times, median; K2 as the evaluator calls it (deterministic, env_actions only).  Rows: one tile per
    SM (18 944), 131 072 and 1 Mi.  With the time, the share of each hardware bound: the MMA work (2 x (32 x 128 + 128 x 128
    + 128 x 16) = 45 056 FLOP per row, zero padding included) over 2 250 TFLOP/s dense bf16, and the HBM bytes (obs 80 B in,
    actions 16 B out per row) over 7.7 TB/s.  The 1 Mi-row observations (80 MB) fit the 126 MB L2 after the first launch.
  * evaluate(): host-clock wall of ppo.PolicyEvaluator.evaluate(), median of 3 after a warm-up, for 16 384 and 65 536
    episodes, the SAC actor and the PPO policy of tools/eval_bench.py in the same call.  The floor rule is off (render = 1)
    and both policies idle the motors (throttle output at -1), so every episode runs to the 402-step time limit.

    python tools/sac_actor_bench.py [--reps 200] [--json out.json]

The card's name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FLOP_PER_ROW = 2 * (32 * 128 + 128 * 128 + 128 * 16)
BYTES_PER_ROW = 20 * 4 + 4 * 4
PEAK_FLOPS, PEAK_BW = 2.25e15, 7.7e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200, help="launches per captured graph")
    ap.add_argument("--json", default=None, help="also write the results to this file")
    args = ap.parse_args()
    import torch

    import __graft_entry__ as ge

    ge.build()
    import fpv_drone_rl_agent_b200 as pkg
    from fpv_drone_rl_agent_b200 import ppo, sac

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    card = card.splitlines()[torch.cuda.current_device()] if card else "unknown"
    print(f"card: {card}")
    dev = torch.device("cuda", torch.cuda.current_device())
    torch.manual_seed(0)
    actor = sac.SacActor(20, 4).to(dev)
    with torch.no_grad():
        actor.mu.bias[3] = -5.0  # tanh -> -1: the motors idle
    packed_sac = sac.PackedSacActor(actor, dev)
    model = ppo.ActorCritic().to(dev)
    with torch.no_grad():
        model.mu.bias[3] = -1.0
    packed_ppo = ppo.PackedPolicy(model, dev)
    stats = ppo.RunningStats(20, dev)
    norm = (stats.mean, stats.inv_std)

    def timed_graph(body):
        g = ppo._capture(body, dev)
        g.replay()
        torch.cuda.synchronize()

        def run():
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            g.replay()
            e.record()
            torch.cuda.synchronize()
            return s.elapsed_time(e) * 1e3 / args.reps
        return run

    kernel_rows = []
    for n in (148 * 128, 131_072, 1 << 20):
        obs = torch.randn(n, 20, device=dev)
        act_s, act_p = torch.empty(n, 4, device=dev), torch.empty(n, 4, device=dev)
        sac.sac_actor_forward(packed_sac, obs, norm=norm, obs_clip=10.0, actions=act_s)  # one-time attribute setup outside capture
        packed_ppo.act(obs, act_p, norm, 10.0)
        run_s = timed_graph(lambda: [sac.sac_actor_forward(packed_sac, obs, norm=norm, obs_clip=10.0, actions=act_s) for _ in range(args.reps)])
        run_p = timed_graph(lambda: [packed_ppo.act(obs, act_p, norm, 10.0) for _ in range(args.reps)])
        ts, tp = [], []
        for _ in range(5):
            ts.append(run_s())
            tp.append(run_p())
        t_s, t_p = statistics.median(ts), statistics.median(tp)
        row = dict(rows=n, sac_us=t_s, sac_rows_per_s=n / (t_s * 1e-6), ppo_us=t_p, ppo_rows_per_s=n / (t_p * 1e-6),
                   sac_mma_share=n * FLOP_PER_ROW / PEAK_FLOPS / (t_s * 1e-6), sac_hbm_share=n * BYTES_PER_ROW / PEAK_BW / (t_s * 1e-6),
                   sac_us_all=ts, ppo_us_all=tp)
        kernel_rows.append(row)
        print(f"{n:8d} rows: SAC actor (K8) {t_s:7.2f} us = {row['sac_rows_per_s']:.3e} rows/s (MMA bound {100 * row['sac_mma_share']:.1f} %, "
              f"HBM bound {100 * row['sac_hbm_share']:.1f} %); PPO forward (K2) {t_p:7.2f} us = {row['ppo_rows_per_s']:.3e} rows/s")
        del obs, act_s, act_p
    cfg = pkg.default_config()
    cfg.update(render=1)
    eval_rows = []
    for n in (16384, 65536):
        row = dict(episodes=n)
        for name, packed in (("sac", packed_sac), ("ppo", packed_ppo)):
            ev = ppo.PolicyEvaluator(packed, stats, cfg, n, seed=1)
            ev.evaluate()  # warm-up (captures the evaluator's graph)
            walls, summary = [], None
            for _ in range(3):
                t0 = time.perf_counter()
                summary, _ = ev.evaluate()
                walls.append(time.perf_counter() - t0)
            row.update({f"{name}_evaluate_ms": 1e3 * statistics.median(walls), f"{name}_evaluate_all_ms": [1e3 * w for w in walls],
                        f"{name}_steps": summary["steps"], f"{name}_mean_ep_length": summary["mean_ep_length"]})
            ev.close()
            torch.cuda.empty_cache()
        eval_rows.append(row)
        print(f"{n:6d} episodes: evaluate() SAC {row['sac_evaluate_ms']:6.1f} ms ({row['sac_steps']} steps, mean length {row['sac_mean_ep_length']:.1f}), "
              f"PPO {row['ppo_evaluate_ms']:6.1f} ms ({row['ppo_steps']} steps, mean length {row['ppo_mean_ep_length']:.1f})")
    result = dict(card=card, reps=args.reps, kernel=kernel_rows, evaluate=eval_rows)
    print(json.dumps(result))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
