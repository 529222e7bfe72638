"""Time GAE + TRPO + critic through the GRU modules on the bandit meta-env batch (config 4 shard) on one GPU.
CELL=lstm runs LstmLinear modules instead; H other than 4 (or CELL=lstm) takes K9's run-time-sized instances."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import relearn_b200 as R

E = int(os.environ.get("E", 131072)); ARMS = int(os.environ.get("ARMS", 2)); N = int(os.environ.get("EPISODES", 10))
H = int(os.environ.get("H", 4)); CELL = os.environ.get("CELL", "gru"); STEPS = int(os.environ.get("CRITIC_STEPS", 80))
T = 2 * N - 1
ctx = R.Context(0)
env = R.build_env(ctx, R.MetaEnv(R.UniformBernoulliBandits(ARMS), N), E, seed=1)
g = (R.LstmLinearConfig if CELL == "lstm" else R.GruLinearConfig)(hidden_dim=H)
init = R.init_lstm_linear_params if CELL == "lstm" else R.init_gru_linear_params
agent = R.ActorCriticConfig(policy_config=R.TrpoConfig(policy_fn_config=g),
                            critic_config=R.ValuesOptConfig(state_value_fn_config=g, opt_steps_per_update=STEPS)).build_agent(env)
rng = np.random.default_rng(0)
agent.policy.policy_fn.set_weights(init(rng, env.num_features, H, ARMS))
agent.critic.state_value_fn.set_weights(init(rng, env.num_features, H, 1))
traj = R.Trajectory(env, T)
res = []
for it in range(4):
    summ = R.rollout(env, agent.actor(), R.HistoryDataBound(T, 0), traj)
    e0 = ctx.event().record()
    adv = agent.critic.advantages(traj)
    e1 = ctx.event().record()
    log = {}
    st = agent.policy.update(traj, adv, log)
    cs = agent.critic.update(traj, log)
    res.append((round(e0.elapsed_ms(e1), 3), round(log["policy/update_time"] * 1e3, 3), round(cs.update_ms, 3), st,
                log["num_backtracks"], log["cg_iterations"], round(summ.step_reward.mean, 4)))
print(f"{CELL} E={E} T={T} H={H} steps={E * T}: adv / policy / critic({STEPS}) ms, status, backtracks, cg, mean reward:", res[1:])
