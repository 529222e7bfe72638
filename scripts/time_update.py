"""Time GAE + TRPO + critic on the cartpole-trpo batch (E=4096, T=256) on one GPU."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import relearn_b200 as R

E = int(os.environ.get("E", 4096)); T = int(os.environ.get("T", 256))
ctx = R.Context(0)
cfg = R.CartPoleConfig().wrap(R.VisibleStepLimit(500))
env = R.build_env(ctx, cfg, E, seed=1)
agent = R.ActorCriticConfig().build_agent(env)
rng = np.random.default_rng(0)
agent.policy.policy_fn.set_weights(R.init_params(rng, 5, 128, 2))
agent.critic.state_value_fn.set_weights(R.init_params(rng, 5, 128, 1))
traj = R.Trajectory(env, T)
res = []
for it in range(4):
    R.rollout(env, agent.actor(), R.HistoryDataBound(T, 0), traj, want_summary=False)
    e0 = ctx.event().record()
    adv = agent.critic.advantages(traj)
    e1 = ctx.event().record()
    log = {}
    st = agent.policy.update(traj, adv, log)
    cs = agent.critic.update(traj, log)
    res.append((e0.elapsed_ms(e1), log["policy/update_time"] * 1e3, cs.update_ms, st, log["num_backtracks"], log["cg_iterations"]))
print("adv/policy/critic ms, status, backtracks, cg:", [tuple(round(x, 3) if isinstance(x, float) else x for x in r) for r in res[1:]])
