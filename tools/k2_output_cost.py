import os, sys, statistics, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as ge; ge.build()
from fpv_drone_rl_agent_b200 import ppo
dev = torch.device('cuda')
m = ppo.ActorCritic().to(dev); pol = ppo.PackedPolicy(m, dev)
def timed(fn, reps=9):
    ts = []
    for _ in range(reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); fn(); e.record(); torch.cuda.synchronize(); ts.append(s.elapsed_time(e))
    return statistics.median(ts) * 1e3
for n in (131072, 1 << 20):
    obs = torch.randn(n, 20, device=dev)
    acts = torch.zeros(n, 4, device=dev); eacts = torch.zeros(n, 4, device=dev); vals = torch.zeros(n, device=dev); logp = torch.zeros(n, device=dev); on = torch.zeros(n, 20, device=dev)
    full = lambda: ppo.policy_forward(pol, obs, seed=1, step=3, actions=acts, env_actions=eacts, values=vals, log_probs=logp, obs_norm=on)
    noon = lambda: ppo.policy_forward(pol, obs, seed=1, step=3, actions=acts, env_actions=eacts, values=vals, log_probs=logp)
    valonly = lambda: ppo.policy_forward(pol, obs, deterministic=True, values=vals)
    for f in (full, noon, valonly): f()
    torch.cuda.synchronize()
    print(n, 'all outputs %.1f us | without obs_norm %.1f us | values only %.1f us' % (timed(full), timed(noon), timed(valonly)))
