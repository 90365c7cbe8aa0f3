"""Deterministic policy evaluation (ppo.PolicyEvaluator, qx_episode_record) on the GPU, for 16 384 and 65 536 episodes with the
floor rule off (render = 1), so that nearly every episode runs to the 402-step time limit:

  * per step, forward + step + record and forward + step alone: CUDA-event time of one captured 32-step chunk from the initial
    state (every record open), the two graphs alternated;
  * the record launch alone (`reps` launches in one captured graph), on the initial state (every record open: a 4 B end word
    and one 16 B state load per env) and after an evaluation (every record closed: the end word only);
  * the wall time of a whole evaluate() call (state restore from the host, chunk replays, one host read per chunk, summary),
    and how many steps it ran.

    python tools/eval_bench.py [--reps 50] [--json out.json]

The policy is a freshly initialised [128, 128] ActorCritic with default observation statistics whose throttle output is
biased to -1: the motors idle, the drone stays on the ground and, with the floor rule off, every episode runs to the 402-step
time limit -- the longest evaluation there is (the policy forward costs the same whatever its weights).  The card's name and
power limit are read in the same run."""
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

CHUNK = 32


def events_us(fn, reps):
    """mean time of `reps` back-to-back calls of fn, in microseconds (CUDA events)"""
    import torch

    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) * 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50, help="back-to-back record launches per timing")
    ap.add_argument("--json", default=None, help="also write the results to this file")
    args = ap.parse_args()
    import torch

    import __graft_entry__ as ge

    ge.build()
    import fpv_drone_rl_agent_b200 as pkg
    from fpv_drone_rl_agent_b200 import ppo

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    card = card.splitlines()[torch.cuda.current_device()] if card else "unknown"
    print(f"card: {card}")
    dev = torch.device("cuda", torch.cuda.current_device())
    torch.manual_seed(0)
    model = ppo.ActorCritic().to(dev)
    with torch.no_grad():
        model.mu.bias[3] = -1.0  # throttle -1: the motors idle and, with the floor rule off, every episode runs to the time limit
    packed = ppo.PackedPolicy(model, dev)
    stats = ppo.RunningStats(20, dev)
    cfg = pkg.default_config()
    cfg.update(render=1)
    rows = []
    for n in (16384, 65536):
        ev = ppo.PolicyEvaluator(packed, stats, cfg, n, seed=1, chunk=CHUNK)
        state0, obs0 = ev.sim.get_state(), ev.obs.clone()

        def restart():
            ev.sim.set_state(state0)
            ev.obs.copy_(obs0)
            for t in (ev.ret, ev.length, ev.end, ev.n_closed):
                t.zero_()

        def capture(record):
            st = torch.cuda.Stream(device=dev)
            st.wait_stream(torch.cuda.current_stream(dev))
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(st), torch.cuda.graph(g, stream=st):
                for _ in range(CHUNK):
                    ppo.policy_forward(packed, ev.obs, norm=ev.norm, obs_clip=ev.obs_clip, deterministic=True, env_actions=ev.env_actions)
                    ev.sim.step(ev.env_actions, ev.obs, ev.reward, ev.te, ev.tr)
                    if record:
                        ev.sim.episode_record(ev.ret, ev.length, ev.end, ev.n_closed)
            torch.cuda.current_stream(dev).wait_stream(st)
            return g

        ev.norm[0].copy_(stats.mean)
        ev.norm[1].copy_(stats.inv_std)
        graphs = {True: capture(True), False: capture(False)}
        t_chunk = {True: [], False: []}
        for _ in range(5):  # alternated, so that a drift of the clock shows in both
            for rec in (True, False):
                restart()
                graphs[rec].replay()  # warm: the chunk's memory in L2 as it would be mid-evaluation
                restart()
                t_chunk[rec].append(events_us(graphs[rec].replay, 1) / CHUNK)
        # the record launch alone: `reps` launches captured in one graph (issued one by one from Python, the host would be timed)
        st = torch.cuda.Stream(device=dev)
        st.wait_stream(torch.cuda.current_stream(dev))
        g_rec = torch.cuda.CUDAGraph()
        with torch.cuda.stream(st), torch.cuda.graph(g_rec, stream=st):
            for _ in range(args.reps):
                ev.sim.episode_record(ev.ret, ev.length, ev.end, ev.n_closed)
        torch.cuda.current_stream(dev).wait_stream(st)
        restart()  # initial state: no episode has ended, every record stays open
        g_rec.replay()
        rec_open = statistics.median(events_us(g_rec.replay, 1) / args.reps for _ in range(5))
        ev.evaluate()  # warm-up (captures the evaluator's own graph)
        walls, summary = [], None
        for _ in range(3):
            t0 = time.perf_counter()
            summary, _ = ev.evaluate()
            walls.append(time.perf_counter() - t0)
        g_rec.replay()
        rec_closed = statistics.median(events_us(g_rec.replay, 1) / args.reps for _ in range(5))  # every record closed
        row = dict(episodes=n, steps_run=summary["steps"], mean_ep_length=summary["mean_ep_length"], success_rate=summary["success_rate"],
                   step_with_record_us=statistics.median(t_chunk[True]), step_without_record_us=statistics.median(t_chunk[False]),
                   record_open_us=rec_open, record_closed_us=rec_closed, evaluate_wall_s=statistics.median(walls), evaluate_wall_all_s=walls)
        row["record_share_of_step"] = rec_open / row["step_with_record_us"]
        rows.append(row)
        print(f"{n:6d} episodes: forward+step+record {row['step_with_record_us']:7.1f} us/step, forward+step {row['step_without_record_us']:7.1f} us/step; "
              f"record alone {rec_open:5.2f} us (open), {rec_closed:5.2f} us (closed) = {100 * row['record_share_of_step']:.1f} % of the step; "
              f"evaluate() {row['evaluate_wall_s'] * 1e3:7.1f} ms wall for {summary['steps']} steps (mean length {summary['mean_ep_length']:.1f}, "
              f"success {summary['success_rate']:.3f})")
        del graphs
        ev.close()
        torch.cuda.empty_cache()
    result = dict(card=card, chunk=CHUNK, reps=args.reps, rows=rows)
    print(json.dumps(result))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
