import os, sys, time, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as ge; ge.build()
from fpv_drone_rl_agent_b200 import ppo
for tf32 in (False, True):
    torch.backends.cuda.matmul.allow_tf32 = tf32
    for graph in (False, True):
        cfg = ppo.PPOConfig(n_envs=16384, n_steps=64, n_epochs=4, batch_size=32768, target_kl=0.0, log_std_init=-1.0, graph_update=graph)
        t = ppo.PPOTrainer(cfg, device="cuda")
        t.learn_iteration(); torch.cuda.synchronize()
        t0 = time.perf_counter(); t.rollout.collect(); torch.cuda.synchronize(); t1 = time.perf_counter()
        t.update(); torch.cuda.synchronize(); t2 = time.perf_counter()
        print(f"tf32={tf32} graph={graph}: rollout {1e3*(t1-t0):.1f} ms, update {1e3*(t2-t1):.1f} ms for 128 minibatch steps = {1e3*(t2-t1)/128:.3f} ms/step")
        t.sim.close()
